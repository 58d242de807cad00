// runtime.cu -- host runtime behind the C ABI in include/frx.h.
//
// Owns: the packed weights (one device arena), the activation workspaces, the
// decoder's KV caches, and the CUDA graphs of the decode loop.  Everything is
// enqueued on the caller's stream.  No CPU fallback: every entry point fails
// loudly if the device or a kernel launch fails.
//
// Reference lines cited are in /root/reference/networks/EfficientSATRN.py.
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <map>
#include <string>
#include <vector>

#include "../../include/frx.h"
#include "kernels.h"
#include "runtime.h"

using namespace frx;

// ---------------------------------------------------------------------------
// helpers
// ---------------------------------------------------------------------------
static int fail(frx_handle* h, const char* fmt, ...) {
  char buf[1024];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  if (h) h->err = buf;
  return 1;
}

#define CK(expr)                                                                          \
  do {                                                                                    \
    cudaError_t e__ = (expr);                                                             \
    if (e__ != cudaSuccess)                                                               \
      return fail(h, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e__), __FILE__, __LINE__); \
  } while (0)

#define CKL()                                                                             \
  do {                                                                                    \
    cudaError_t e__ = cudaGetLastError();                                                 \
    if (e__ != cudaSuccess)                                                               \
      return fail(h, "kernel launch failed: %s (%s:%d)", cudaGetErrorString(e__), __FILE__, __LINE__); \
    h->launches++;                                                                        \
  } while (0)

// Every ABI call runs on the handle's device and puts the caller's current device back on return (torch keeps its own
// notion of the current device; silently changing it would redirect the caller's later allocations and launches).
struct DeviceGuard {
  int prev = -1;
  bool changed = false;
  cudaError_t enter(int dev) {
    cudaError_t e = cudaGetDevice(&prev);
    if (e != cudaSuccess) return e;
    if (prev != dev) {
      e = cudaSetDevice(dev);
      changed = e == cudaSuccess;
    }
    return e;
  }
  ~DeviceGuard() {
    if (changed) cudaSetDevice(prev);
  }
};
#define ON_DEVICE(dev) \
  DeviceGuard guard__;  \
  CK(guard__.enter(dev))

static int dev_alloc(frx_handle* h, void** p, size_t bytes) {
  if (bytes == 0) bytes = 256;
  cudaError_t e = cudaMalloc(p, bytes);
  if (e != cudaSuccess) return fail(h, "cudaMalloc(%zu) failed: %s", bytes, cudaGetErrorString(e));
  h->allocs.push_back(*p);
  h->device_bytes += (int64_t)bytes;
  return 0;
}

// ---------------------------------------------------------------------------
// weight arena: packed on the host, uploaded once
// ---------------------------------------------------------------------------
struct ArenaBuilder {
  std::vector<float> host;
  size_t add(const float* src, size_t n) {
    size_t off = (host.size() + 63) / 64 * 64;
    host.resize(off + n);
    if (src) memcpy(host.data() + off, src, n * sizeof(float));
    return off;
  }
  float* at(size_t off) { return host.data() + off; }
};

static const HostTensor* find(frx_handle* h, const std::string& name) {
  auto it = h->raw.find(name);
  return it == h->raw.end() ? nullptr : &it->second;
}

static int need(frx_handle* h, const std::string& name, std::initializer_list<int64_t> shape,
                const HostTensor** out) {
  const HostTensor* t = find(h, name);
  if (!t) return fail(h, "missing tensor '%s'", name.c_str());
  std::vector<int64_t> s(shape);
  if (t->shape != s) {
    std::string got, want;
    for (auto v : t->shape) got += std::to_string(v) + ",";
    for (auto v : s) want += std::to_string(v) + ",";
    return fail(h, "tensor '%s' has shape [%s] expected [%s]", name.c_str(), got.c_str(), want.c_str());
  }
  *out = t;
  return 0;
}

// eval-mode BatchNorm folded to y = x*alpha + beta, computed like ATen's CPU path
// (invstd = 1/sqrt(var+eps); alpha = w*invstd; beta = b - mean*alpha).
static int fold_bn(frx_handle* h, ArenaBuilder& ab, const std::string& p, int C, float eps,
                   const float* conv_bias, size_t* off_scale, size_t* off_shift) {
  const HostTensor *w, *b, *mu, *var;
  if (need(h, p + ".weight", {C}, &w) || need(h, p + ".bias", {C}, &b) ||
      need(h, p + ".running_mean", {C}, &mu) || need(h, p + ".running_var", {C}, &var))
    return 1;
  *off_scale = ab.add(nullptr, C);
  *off_shift = ab.add(nullptr, C);
  for (int c = 0; c < C; ++c) {
    float invstd = 1.0f / sqrtf(var->f[c] + eps);
    float alpha = w->f[c] * invstd;
    float beta = b->f[c] - mu->f[c] * alpha;
    if (conv_bias) beta += conv_bias[c] * alpha;
    ab.at(*off_scale)[c] = alpha;
    ab.at(*off_shift)[c] = beta;
  }
  return 0;
}

// conv weight [O][I][kh][kw] -> [O][kh][kw][I]  (K index = (kh*KW+kw)*I + i)
static int pack_conv(frx_handle* h, ArenaBuilder& ab, const std::string& name, int O, int I, int k,
                     size_t* off) {
  const HostTensor* w;
  if (need(h, name, {O, I, k, k}, &w)) return 1;
  *off = ab.add(nullptr, (size_t)O * I * k * k);
  float* d = ab.at(*off);
  for (int o = 0; o < O; ++o)
    for (int i = 0; i < I; ++i)
      for (int t = 0; t < k * k; ++t) d[((size_t)o * k * k + t) * I + i] = w->f[((size_t)o * I + i) * k * k + t];
  return 0;
}

// depthwise weight [C][1][3][3] -> [9][C]
static int pack_dw(frx_handle* h, ArenaBuilder& ab, const std::string& name, int C, size_t* off) {
  const HostTensor* w;
  if (need(h, name, {C, 1, 3, 3}, &w)) return 1;
  *off = ab.add(nullptr, (size_t)9 * C);
  float* d = ab.at(*off);
  for (int c = 0; c < C; ++c)
    for (int t = 0; t < 9; ++t) d[(size_t)t * C + c] = w->f[(size_t)c * 9 + t];
  return 0;
}

// linear weight [N][K] placed transposed into a [K][Ntot] matrix at column col0
static void put_transposed(float* dst, int Ntot, int col0, const float* w, int N, int K) {
  for (int n = 0; n < N; ++n)
    for (int k = 0; k < K; ++k) dst[(size_t)k * Ntot + col0 + n] = w[(size_t)n * K + k];
}

static void same_pad(int in, int k, int stride, int* out, int* pad_lo) {
  // timm 0.4.9 layers/padding.py: static symmetric for stride 1, TF dynamic for stride 2
  *out = (in + stride - 1) / stride;
  if (stride == 1) { *pad_lo = (k - 1) / 2; return; }
  int pad = (*out - 1) * stride + k - in;
  if (pad < 0) pad = 0;
  *pad_lo = pad / 2;
}

// (kind, repeats, kernel, stride, expand, out_ch, se_ratio_x100)  -- SURVEY App. A.1
static const int kArch[6][7] = {
    {0, 2, 3, 1, 1, 24, 0},  {1, 4, 3, 2, 4, 48, 0},    {1, 4, 3, 2, 4, 64, 0},
    {2, 6, 3, 2, 4, 128, 25}, {2, 9, 3, 1, 6, 160, 25}, {2, 15, 3, 2, 6, 256, 25}};

// ---------------------------------------------------------------------------
// C ABI
// ---------------------------------------------------------------------------
extern "C" const char* frx_version(void) { return "frx 0.1 sm_100a"; }

extern "C" const char* frx_last_error(const frx_handle* h) { return h ? h->err.c_str() : "null handle"; }

extern "C" int frx_create(const frx_config* cfg, frx_handle** out) {
  if (!cfg || !out) return 1;
  frx_handle* h = new frx_handle();
  h->cfg = *cfg;
  *out = h;
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0)
    return fail(h, "no CUDA device available (%s): frx has no CPU fallback", cudaGetErrorString(e));
  if (cfg->device < 0 || cfg->device >= ndev) return fail(h, "device %d out of range", cfg->device);
  ON_DEVICE(cfg->device);
  cudaDeviceProp prop;
  CK(cudaGetDeviceProperties(&prop, cfg->device));
  if (prop.major != 10) return fail(h, "device is sm_%d%d; frx is built for sm_100a (B200) only", prop.major, prop.minor);
  h->num_sms = prop.multiProcessorCount;
  if (cfg->network != FRX_NET_EFFICIENT_SATRN && cfg->network != FRX_NET_LITE_SATRN && cfg->network != FRX_NET_SWIN)
    return fail(h, "unknown network %d", cfg->network);
  if (cfg->network == FRX_NET_SWIN && (cfg->height != 384 || cfg->width != 384 || cfg->in_ch != 3 || cfg->enc_hidden != 1024))
    return fail(h, "SWIN is fixed to Swin-B/384: 384x384x3 input, 1024-wide memory (networks/SWIN.py:1028-1031)");
  if (cfg->dec_hidden % cfg->dec_heads || (cfg->dec_hidden / cfg->dec_heads != 32 && cfg->dec_hidden / cfg->dec_heads != 64))
    return fail(h, "decoder head_dim must be 32 or 64");
  if (cfg->dec_hidden > 512) return fail(h, "decoder hidden_dim > 512 not supported");
  if (cfg->max_batch <= 0 || cfg->max_steps <= 0) return fail(h, "max_batch/max_steps must be positive");
  return 0;
}

extern "C" void frx_destroy(frx_handle* h) {
  if (!h) return;
  DeviceGuard guard;
  guard.enter(h->cfg.device);
  frx_train_destroy(h);
  for (auto& kv : h->graphs) cudaGraphExecDestroy(kv.second.exec);
  for (void* p : h->allocs) cudaFree(p);
  for (auto& kv : h->taps) cudaFree(kv.second.data);
  if (h->ev[0]) for (int i = 0; i < 5; ++i) cudaEventDestroy(h->ev[i]);
  for (auto& sl : h->pipe) {
    if (sl.h2d) { cudaEventDestroy(sl.h2d); cudaEventDestroy(sl.enc); cudaEventDestroy(sl.done); cudaEventDestroy(sl.d2h); }
  }
  if (h->pipe_h2d) { cudaStreamDestroy(h->pipe_h2d); cudaStreamDestroy(h->pipe_d2h); cudaStreamDestroy(h->pipe_enc); }
  delete h;
}

extern "C" int frx_load_tensor(frx_handle* h, const char* name, const void* data, const int64_t* shape,
                               int32_t ndim, int32_t dtype) {
  if (!h || !name || !data) return fail(h, "frx_load_tensor: null argument");
  HostTensor t;
  size_t n = 1;
  for (int i = 0; i < ndim; ++i) { t.shape.push_back(shape[i]); n *= (size_t)shape[i]; }
  if (dtype == FRX_DTYPE_F32) {
    t.f.resize(n);
    CK(cudaMemcpy(t.f.data(), data, n * sizeof(float), cudaMemcpyDefault));
  } else if (dtype == FRX_DTYPE_I64) {
    std::vector<int64_t> tmp(n);
    CK(cudaMemcpy(tmp.data(), data, n * sizeof(int64_t), cudaMemcpyDefault));
    t.f.resize(n);
    for (size_t i = 0; i < n; ++i) t.f[i] = (float)tmp[i];
  } else {
    return fail(h, "frx_load_tensor('%s'): unsupported dtype %d", name, dtype);
  }
  h->raw[name] = std::move(t);
  h->finalized = false;
  return 0;
}

extern "C" int frx_set_option(frx_handle* h, const char* key, int64_t value) {
  if (!h || !key) return 1;
  ON_DEVICE(h->cfg.device);
  std::string k(key);
  if (k == "taps") h->opt_taps = value != 0;
  else if (k == "graphs") h->opt_graphs = value != 0;
  else if (k == "step16") h->opt_step16 = value != 0;
  else if (k == "pipe_enc") h->opt_pipe_enc = value != 0;   // pipelined host entry: next batch's encoder on its own stream
  else if (k == "timing") h->opt_timing = value != 0;
  else if (k == "cluster_images") {}  // accepted for compatibility: clusters always own 8 images
  else if (k == "dec_hpc") h->opt_dec_hpc = (value == 1 || value == 2) ? (int)value : 0;  // heads per CTA of the 256-wide decode kernel, 0 = by batch size
  else if (k == "conv24") h->opt_conv24 = value != 0;  // 0: stage-0 convs through the tcgen05 im2col GEMM instead
  else if (k == "enc_fp32") h->opt_enc_fp32 = value != 0;
  else if (k == "tc_ws") h->opt_tc_ws = value != 0;
  else if (k == "train_splitk") h->opt_train_splitk = value != 0;  // 0: every training GEMM reduces K in one CTA pass (the summation order of the r2 parity runs)
  else if (k == "tc_im2col") h->opt_tc_im2col = value != 0;
  else if (k == "prof") {
    h->opt_prof = value != 0;
    if (h->opt_prof && !h->prof) { void* p; if (dev_alloc(h, &p, 16 * 8)) return 1; h->prof = (long long*)p; }
  }
  else if (k == "parts") {
    // the workspaces are sized for the parts chosen at the first finalize: a later change would leave them missing
    if (h->ws_ready && ((int)value & 3) != h->opt_parts)
      return fail(h, "option 'parts' cannot change after the first frx_finalize_weights (create a new handle)");
    h->opt_parts = (int)value & 3;
    h->finalized = false;
  }
  else return fail(h, "unknown option '%s'", key);
  return 0;
}

extern "C" int64_t frx_launch_count(const frx_handle* h) { return h ? h->launches : 0; }
extern "C" int64_t frx_device_bytes(const frx_handle* h) { return h ? h->device_bytes : 0; }

extern "C" int frx_read_prof(frx_handle* h, int64_t* out16) {
  if (!h || !out16 || !h->prof) return fail(h, "profiling not enabled (frx_set_option(h, \"prof\", 1))");
  ON_DEVICE(h->cfg.device);
  CK(cudaMemcpy(out16, h->prof, 16 * 8, cudaMemcpyDeviceToHost));
  return 0;
}

extern "C" int frx_last_timing(const frx_handle* h, float* ms4) {
  if (!h || !ms4) return 1;
  for (int i = 0; i < 4; ++i) ms4[i] = h->last_ms[i];
  return 0;
}

// ---------------------------------------------------------------------------
// finalize: pack weights, allocate workspaces
// ---------------------------------------------------------------------------
static int pack_trunk_efficientnet(frx_handle* h, ArenaBuilder& ab) {
  const frx_config& c = h->cfg;
  const std::string e = "encoder.shallow_cnn.";
  const HostTensor* w;
  if (need(h, e + "conv_stem.weight", {24, c.in_ch, 3, 3}, &w)) return 1;
  h->stem_w = ab.add(w->f.data(), w->f.size());
  if (fold_bn(h, ab, e + "bn1", 24, 1e-3f, nullptr, &h->stem_sc, &h->stem_sh)) return 1;
  int cin = 24;
  h->blocks.clear();
  for (int s = 0; s < 6; ++s) {
    for (int r = 0; r < kArch[s][1]; ++r) {
      BlockW b{};
      b.kind = kArch[s][0];
      b.k = kArch[s][2];
      b.stride = r == 0 ? kArch[s][3] : 1;
      b.cin = cin;
      b.cout = kArch[s][5];
      b.mid = cin * kArch[s][4];
      b.se_r = cin * kArch[s][6] / 100;
      b.residual = (b.cin == b.cout && b.stride == 1);
      std::string p = e + "eff_block." + std::to_string(s) + "." + std::to_string(r);
      b.name = "eff_block." + std::to_string(s) + "." + std::to_string(r);
      if (b.kind == 0) {
        if (pack_conv(h, ab, p + ".conv.weight", b.cout, b.cin, b.k, &b.w_a)) return 1;
        if (fold_bn(h, ab, p + ".bn1", b.cout, 1e-3f, nullptr, &b.sc_a, &b.sh_a)) return 1;
      } else if (b.kind == 1) {
        if (pack_conv(h, ab, p + ".conv_exp.weight", b.mid, b.cin, b.k, &b.w_a)) return 1;
        if (fold_bn(h, ab, p + ".bn1", b.mid, 1e-3f, nullptr, &b.sc_a, &b.sh_a)) return 1;
        if (pack_conv(h, ab, p + ".conv_pwl.weight", b.cout, b.mid, 1, &b.w_b)) return 1;
        if (fold_bn(h, ab, p + ".bn2", b.cout, 1e-3f, nullptr, &b.sc_b, &b.sh_b)) return 1;
      } else {
        if (pack_conv(h, ab, p + ".conv_pw.weight", b.mid, b.cin, 1, &b.w_a)) return 1;
        if (fold_bn(h, ab, p + ".bn1", b.mid, 1e-3f, nullptr, &b.sc_a, &b.sh_a)) return 1;
        if (pack_dw(h, ab, p + ".conv_dw.weight", b.mid, &b.w_dw)) return 1;
        if (fold_bn(h, ab, p + ".bn2", b.mid, 1e-3f, nullptr, &b.sc_dw, &b.sh_dw)) return 1;
        const HostTensor *w1, *b1, *w2, *b2;
        if (need(h, p + ".se.conv_reduce.weight", {b.se_r, b.mid, 1, 1}, &w1) ||
            need(h, p + ".se.conv_reduce.bias", {b.se_r}, &b1) ||
            need(h, p + ".se.conv_expand.weight", {b.mid, b.se_r, 1, 1}, &w2) ||
            need(h, p + ".se.conv_expand.bias", {b.mid}, &b2))
          return 1;
        b.se_w1 = ab.add(w1->f.data(), w1->f.size());
        b.se_b1 = ab.add(b1->f.data(), b1->f.size());
        b.se_w2 = ab.add(w2->f.data(), w2->f.size());
        b.se_w2t = ab.add(nullptr, w2->f.size());  // [R][C] for the bf16 path's coalesced reads
        for (int cc = 0; cc < b.mid; ++cc)
          for (int rr = 0; rr < b.se_r; ++rr) ab.at(b.se_w2t)[(size_t)rr * b.mid + cc] = w2->f[(size_t)cc * b.se_r + rr];
        b.se_b2 = ab.add(b2->f.data(), b2->f.size());
        if (pack_conv(h, ab, p + ".conv_pwl.weight", b.cout, b.mid, 1, &b.w_b)) return 1;
        if (fold_bn(h, ab, p + ".bn3", b.cout, 1e-3f, nullptr, &b.sc_b, &b.sh_b)) return 1;
      }
      h->blocks.push_back(b);
      cin = b.cout;
    }
  }
  if (pack_conv(h, ab, e + "conv_last.weight", c.enc_hidden, 256, 1, &h->last_w)) return 1;
  if (fold_bn(h, ab, e + "bn2", c.enc_hidden, 1e-5f, nullptr, &h->last_sc, &h->last_sh)) return 1;
  return 0;
}

static int pack_trunk_lite(frx_handle* h, ArenaBuilder& ab) {
  // LiteSATRN.py:21-70: 4 x (conv3x3 p1 no-bias, BN, ReLU, maxpool2)
  const frx_config& c = h->cfg;
  const std::string e = "encoder.shallow_cnn.";
  int H = c.enc_hidden;
  int chans[4][2] = {{c.in_ch, H / 2}, {H / 2, H}, {H, H}, {H, H}};
  for (int i = 0; i < 4; ++i) {
    LiteConvW& L = h->lite[i];
    L.cin = chans[i][0];
    L.cout = chans[i][1];
    if (i == 0) {
      const HostTensor* w;
      if (need(h, e + "conv0.weight", {L.cout, L.cin, 3, 3}, &w)) return 1;
      L.w = ab.add(w->f.data(), w->f.size());  // direct kernel uses [O][I][3][3]
    } else if (pack_conv(h, ab, e + "conv" + std::to_string(i) + ".weight", L.cout, L.cin, 3, &L.w)) {
      return 1;
    }
    if (fold_bn(h, ab, e + "batch_norm" + std::to_string(i), L.cout, 1e-5f, nullptr, &L.sc, &L.sh)) return 1;
  }
  return 0;
}

// SwinTRN encoder (networks/SWIN.py:590-741): Swin-B/384, patch 4, window 12, depths 2-2-18-2, heads 4-8-16-32.
static int pack_swin(frx_handle* h, ArenaBuilder& ab) {
  const std::string e = "encoder.";
  const int E = 128, R0 = 96, WS = 12;
  const int depths[4] = {2, 2, 18, 2}, heads[4] = {4, 8, 16, 32};
  auto vec = [&](const std::string& name, std::initializer_list<int64_t> shape, size_t* off) -> int {
    const HostTensor* t;
    if (need(h, name, shape, &t)) return 1;
    *off = ab.add(t->f.data(), t->f.size());
    return 0;
  };
  if (vec(e + "patch_embed.proj.weight", {E, 3, 4, 4}, &h->sw_pe_w) || vec(e + "patch_embed.proj.bias", {E}, &h->sw_pe_b) ||
      vec(e + "patch_embed.norm.weight", {E}, &h->sw_pe_g) || vec(e + "patch_embed.norm.bias", {E}, &h->sw_pe_beta) ||
      vec(e + "absolute_pos_embed", {1, R0 * R0, E}, &h->sw_ape) || vec(e + "norm.weight", {8 * E}, &h->sw_norm_g) ||
      vec(e + "norm.bias", {8 * E}, &h->sw_norm_b))
    return 1;
  h->sw_blocks.clear();
  h->sw_merges.clear();
  for (int i = 0; i < 4; ++i) {
    const int dim = E << i, res = R0 >> i;
    for (int j = 0; j < depths[i]; ++j) {
      SwinBlockW b{};
      b.dim = dim; b.res = res; b.heads = heads[i];
      b.ws = WS; b.shift = (j % 2 == 0) ? 0 : WS / 2;
      if (res <= WS) { b.ws = res; b.shift = 0; }  // :262-265
      const std::string p = e + "layers." + std::to_string(i) + ".blocks." + std::to_string(j) + ".";
      const int T = (2 * b.ws - 1) * (2 * b.ws - 1);
      if (vec(p + "norm1.weight", {dim}, &b.n1_g) || vec(p + "norm1.bias", {dim}, &b.n1_b) ||
          vec(p + "attn.relative_position_bias_table", {T, b.heads}, &b.bias_table) ||
          vec(p + "attn.qkv.weight", {3 * dim, dim}, &b.qkv_w) || vec(p + "attn.qkv.bias", {3 * dim}, &b.qkv_b) ||
          vec(p + "attn.proj.weight", {dim, dim}, &b.proj_w) || vec(p + "attn.proj.bias", {dim}, &b.proj_b) ||
          vec(p + "norm2.weight", {dim}, &b.n2_g) || vec(p + "norm2.bias", {dim}, &b.n2_b) ||
          vec(p + "mlp.fc1.weight", {4 * dim, dim}, &b.fc1_w) || vec(p + "mlp.fc1.bias", {4 * dim}, &b.fc1_b) ||
          vec(p + "mlp.fc2.weight", {dim, 4 * dim}, &b.fc2_w) || vec(p + "mlp.fc2.bias", {dim}, &b.fc2_b))
        return 1;
      h->sw_blocks.push_back(b);
    }
    if (i < 3) {
      SwinMergeW m{};
      m.dim = dim; m.res = res;
      const std::string p = e + "layers." + std::to_string(i) + ".downsample.";
      if (vec(p + "reduction.weight", {2 * dim, 4 * dim}, &m.red_w) || vec(p + "norm.weight", {4 * dim}, &m.n_g) ||
          vec(p + "norm.bias", {4 * dim}, &m.n_b))
        return 1;
      h->sw_merges.push_back(m);
    }
  }
  return 0;
}

static int pack_encoder(frx_handle* h, ArenaBuilder& ab) {
  const frx_config& c = h->cfg;
  const int C = c.enc_hidden, F = c.enc_filter;
  const std::string pe = "encoder.positional_encoding.";
  const HostTensor *w0, *b0, *w1, *b1, *th, *tw;
  if (need(h, pe + "dense0.weight", {C / 2, C}, &w0) || need(h, pe + "dense0.bias", {C / 2}, &b0) ||
      need(h, pe + "dense1.weight", {2 * C, C / 2}, &w1) || need(h, pe + "dense1.bias", {2 * C}, &b1) ||
      need(h, "pe2d.h", {h->feat_h, C}, &th) || need(h, "pe2d.w", {h->feat_w, C}, &tw))
    return 1;
  h->pe_w0 = ab.add(w0->f.data(), w0->f.size());
  h->pe_b0 = ab.add(b0->f.data(), b0->f.size());
  h->pe_w1 = ab.add(w1->f.data(), w1->f.size());
  h->pe_b1 = ab.add(b1->f.data(), b1->f.size());
  h->pe_h = ab.add(th->f.data(), th->f.size());
  h->pe_w = ab.add(tw->f.data(), tw->f.size());
  h->enc.clear();
  for (int i = 0; i < c.enc_layers; ++i) {
    EncLayerW L{};
    std::string p = "encoder.attention_layers." + std::to_string(i) + ".";
    const HostTensor *g, *b, *wq, *bq, *wk, *bk, *wv, *bv, *wo, *bo, *dwb;
    if (need(h, p + "norm.weight", {C}, &g) || need(h, p + "norm.bias", {C}, &b)) return 1;
    L.ln_g = ab.add(g->f.data(), C);
    L.ln_b = ab.add(b->f.data(), C);
    std::string a = p + "attention_layer.";
    if (need(h, a + "q_linear.weight", {C, C}, &wq) || need(h, a + "q_linear.bias", {C}, &bq) ||
        need(h, a + "k_linear.weight", {C, C}, &wk) || need(h, a + "k_linear.bias", {C}, &bk) ||
        need(h, a + "v_linear.weight", {C, C}, &wv) || need(h, a + "v_linear.bias", {C}, &bv) ||
        need(h, a + "out_linear.weight", {C, C}, &wo) || need(h, a + "out_linear.bias", {C}, &bo))
      return 1;
    L.w_qkv = ab.add(nullptr, (size_t)3 * C * C);  // [3C][C] : q rows, k rows, v rows
    memcpy(ab.at(L.w_qkv), wq->f.data(), (size_t)C * C * 4);
    memcpy(ab.at(L.w_qkv) + (size_t)C * C, wk->f.data(), (size_t)C * C * 4);
    memcpy(ab.at(L.w_qkv) + (size_t)2 * C * C, wv->f.data(), (size_t)C * C * 4);
    L.b_qkv = ab.add(nullptr, 3 * C);
    memcpy(ab.at(L.b_qkv), bq->f.data(), C * 4);
    memcpy(ab.at(L.b_qkv) + C, bk->f.data(), C * 4);
    memcpy(ab.at(L.b_qkv) + 2 * C, bv->f.data(), C * 4);
    L.w_o = ab.add(wo->f.data(), (size_t)C * C);
    L.b_o = ab.add(bo->f.data(), C);
    if (pack_conv(h, ab, p + "conv0.weight", F, C, 1, &L.w_c0)) return 1;
    if (fold_bn(h, ab, p + "norm0", F, 1e-5f, nullptr, &L.sc_c0, &L.sh_c0)) return 1;
    if (pack_dw(h, ab, p + "depthwise.weight", F, &L.w_dw)) return 1;
    if (need(h, p + "depthwise.bias", {F}, &dwb)) return 1;
    if (fold_bn(h, ab, p + "depthwise_norm", F, 1e-5f, dwb->f.data(), &L.sc_dw, &L.sh_dw)) return 1;
    if (pack_conv(h, ab, p + "conv1.weight", C, F, 1, &L.w_c1)) return 1;
    if (fold_bn(h, ab, p + "norm1", C, 1e-5f, nullptr, &L.sc_c1, &L.sh_c1)) return 1;
    h->enc.push_back(L);
  }
  return 0;
}

static int pack_decoder(frx_handle* h, ArenaBuilder& ab) {
  const frx_config& c = h->cfg;
  const int D = c.dec_hidden, F = c.dec_filter, S = c.dec_src, V = c.num_classes, L = c.dec_layers;
  const HostTensor *emb, *pe, *gw, *gb;
  if (need(h, "decoder.embedding.weight", {V + 1, D}, &emb) || need(h, "pe1d", {500, D}, &pe) ||
      need(h, "decoder.generator.weight", {V, D}, &gw) || need(h, "decoder.generator.bias", {V}, &gb))
    return 1;
  h->emb = ab.add(emb->f.data(), emb->f.size());
  h->pe1d = ab.add(pe->f.data(), pe->f.size());
  h->gen_w = ab.add(gw->f.data(), gw->f.size());  // [V][D] for the teacher-forced GEMM
  h->gen_b = ab.add(gb->f.data(), gb->f.size());
  struct Lin { const HostTensor *w, *b; };
  std::vector<std::map<std::string, Lin>> lw(L);
  h->dec.assign(L, DecLayerW{});
  for (int l = 0; l < L; ++l) {
    std::string p = "decoder.attention_layers." + std::to_string(l) + ".";
    auto lin = [&](const std::string& key, const std::string& name, int N, int K) -> int {
      Lin x;
      if (need(h, p + name + ".weight", {N, K}, &x.w) || need(h, p + name + ".bias", {N}, &x.b)) return 1;
      lw[l][key] = x;
      return 0;
    };
    if (lin("sq", "self_attention_layer.q_linear", D, D) || lin("sk", "self_attention_layer.k_linear", D, D) ||
        lin("sv", "self_attention_layer.v_linear", D, D) || lin("so", "self_attention_layer.out_linear", D, D) ||
        lin("cq", "attention_layer.q_linear", D, D) || lin("ck", "attention_layer.k_linear", D, S) ||
        lin("cv", "attention_layer.v_linear", D, S) || lin("co", "attention_layer.out_linear", D, D) ||
        lin("f0", "feedforward_layer.linear0", F, D) || lin("f1", "feedforward_layer.linear1", D, F))
      return 1;
    DecLayerW& W = h->dec[l];
    auto ln = [&](const std::string& name, size_t* g, size_t* b) -> int {
      const HostTensor *tg, *tb;
      if (need(h, p + name + ".weight", {D}, &tg) || need(h, p + name + ".bias", {D}, &tb)) return 1;
      *g = ab.add(tg->f.data(), D);
      *b = ab.add(tb->f.data(), D);
      return 0;
    };
    if (ln("self_attention_norm", &W.ln1_g, &W.ln1_b) || ln("attention_norm", &W.ln2_g, &W.ln2_b) ||
        ln("feedforward_norm", &W.ln3_g, &W.ln3_b))
      return 1;
    auto tr = [&](const std::string& key, int N, int K, size_t* wo, size_t* bo) {
      *wo = ab.add(nullptr, (size_t)N * K);
      put_transposed(ab.at(*wo), N, 0, lw[l][key].w->f.data(), N, K);
      *bo = ab.add(lw[l][key].b->f.data(), N);
    };
    tr("so", D, D, &W.wt_o, &W.b_o);
    tr("cq", D, D, &W.wt_q2, &W.b_q2);
    tr("co", D, D, &W.wt_o2, &W.b_o2);
    tr("f0", F, D, &W.wt_f0, &W.b_f0);
    tr("f1", D, F, &W.wt_f1, &W.b_f1);
    // row-major copies for the teacher-forced path (igemm wants [N][K])
    W.w_o = ab.add(lw[l]["so"].w->f.data(), (size_t)D * D);
    W.w_q2 = ab.add(lw[l]["cq"].w->f.data(), (size_t)D * D);
    W.w_o2 = ab.add(lw[l]["co"].w->f.data(), (size_t)D * D);
    W.w_f0 = ab.add(lw[l]["f0"].w->f.data(), (size_t)F * D);
    W.w_f1 = ab.add(lw[l]["f1"].w->f.data(), (size_t)D * F);
    W.w_sqkv = ab.add(nullptr, (size_t)3 * D * D);
    memcpy(ab.at(W.w_sqkv), lw[l]["sq"].w->f.data(), (size_t)D * D * 4);
    memcpy(ab.at(W.w_sqkv) + (size_t)D * D, lw[l]["sk"].w->f.data(), (size_t)D * D * 4);
    memcpy(ab.at(W.w_sqkv) + (size_t)2 * D * D, lw[l]["sv"].w->f.data(), (size_t)D * D * 4);
    W.b_sqkv = ab.add(nullptr, 3 * D);
    memcpy(ab.at(W.b_sqkv), lw[l]["sq"].b->f.data(), D * 4);
    memcpy(ab.at(W.b_sqkv) + D, lw[l]["sk"].b->f.data(), D * 4);
    memcpy(ab.at(W.b_sqkv) + 2 * D, lw[l]["sv"].b->f.data(), D * 4);
  }
  // fused step GEMMs: F_0 = [q0 k0 v0]; F_l = [k_{l-1} v_{l-1} q_l k_l v_l]; F_L = [k_{L-1} v_{L-1} gen]
  h->fused.assign(L + 1, FusedW{});
  for (int l = 0; l <= L; ++l) {
    FusedW& Fw = h->fused[l];
    int N = (l == 0 ? 0 : 2 * D) + (l < L ? 3 * D : V);
    Fw.N = N;
    Fw.wt = ab.add(nullptr, (size_t)D * N);
    Fw.b = ab.add(nullptr, N);
    float* wt = ab.at(Fw.wt);
    float* bb = ab.at(Fw.b);
    int col = 0;
    auto put = [&](const HostTensor* w, const HostTensor* b, int n) {
      put_transposed(wt, N, col, w->f.data(), n, D);
      memcpy(bb + col, b->f.data(), n * 4);
      col += n;
    };
    if (l > 0) { put(lw[l - 1]["sk"].w, lw[l - 1]["sk"].b, D); put(lw[l - 1]["sv"].w, lw[l - 1]["sv"].b, D); }
    if (l < L) { put(lw[l]["sq"].w, lw[l]["sq"].b, D); put(lw[l]["sk"].w, lw[l]["sk"].b, D); put(lw[l]["sv"].w, lw[l]["sv"].b, D); }
    else put(gw, gb, V);
  }
  // cross-attention K/V of the encoder memory: one [L*2*D][S] matrix (k_l rows then v_l rows)
  h->w_cross = ab.add(nullptr, (size_t)L * 2 * D * S);
  h->b_cross = ab.add(nullptr, (size_t)L * 2 * D);
  for (int l = 0; l < L; ++l) {
    memcpy(ab.at(h->w_cross) + (size_t)(l * 2) * D * S, lw[l]["ck"].w->f.data(), (size_t)D * S * 4);
    memcpy(ab.at(h->w_cross) + (size_t)(l * 2 + 1) * D * S, lw[l]["cv"].w->f.data(), (size_t)D * S * 4);
    memcpy(ab.at(h->b_cross) + (size_t)(l * 2) * D, lw[l]["ck"].b->f.data(), D * 4);
    memcpy(ab.at(h->b_cross) + (size_t)(l * 2 + 1) * D, lw[l]["cv"].b->f.data(), D * 4);
  }
  return 0;
}

static inline uint32_t bf16_bits(float f) {  // round-to-nearest-even, like __float2bfloat16_rn
  uint32_t u;
  memcpy(&u, &f, 4);
  if ((u & 0x7fffffffu) > 0x7f800000u) return 0x7fc0u;
  u += 0x7fffu + ((u >> 16) & 1u);
  return u >> 16;
}

// host-side fp32 -> 16-bit conversion of ENCODER-side operands (eh_t of common.cuh): IEEE fp16, round-to-nearest-even,
// saturating like cvt.rn.satfinite; or bf16 when the library is built with -DFRX_ENC_FP16=0
static inline uint32_t eh_bits(float f) {
#if FRX_ENC_FP16
  uint32_t u;
  memcpy(&u, &f, 4);
  const uint32_t sign = (u >> 16) & 0x8000u;
  const uint32_t a = u & 0x7fffffffu;
  if (a > 0x7f800000u) return sign | 0x7e00u;              // NaN
  if (a >= 0x477ff000u) return sign | 0x7bffu;             // >= 65520 rounds past the largest finite half: saturate
  if (a < 0x33000001u) return sign;                        // < 2^-25 (or exactly 2^-25, a tie to even 0): zero
  const int e = (int)(a >> 23) - 127;
  uint32_t m = (a & 0x7fffffu) | 0x800000u;                // 24-bit significand
  int shift = e >= -14 ? 13 : 13 + (-14 - e);              // bits dropped (subnormal halves drop more)
  uint32_t q = m >> shift;
  const uint32_t rem = m & ((1u << shift) - 1u), half = 1u << (shift - 1);
  if (rem > half || (rem == half && (q & 1u))) ++q;
  if (e >= -14) return sign | (uint32_t)(((e + 15) << 10) + (q - 0x400u));   // a carry out of q bumps the exponent
  return sign | q;                                         // subnormal (q = 0x400 becomes the smallest normal)
#else
  return bf16_bits(f);
#endif
}

// B-fragment order of mma.m16n8k16 for the persistent decode kernel:
// [cta r][tile][k-pair kp][lane] -> uint4 {b0b1(k-step 2kp), b2b3(2kp), b0b1(2kp+1), b2b3(2kp+1)}.
// rowptr(r, tile, gid) returns the K-float weight row of output column (tile, gid) of CTA r, or nullptr.
template <class F>
static size_t pack_frag_stage(ArenaBuilder& ab, int CL, int NT, int K, F rowptr) {
  const int KP = K / 32;
  size_t off = ab.add(nullptr, (size_t)CL * NT * KP * 32 * 4);
  uint32_t* d = reinterpret_cast<uint32_t*>(ab.at(off));
  for (int r = 0; r < CL; ++r)
    for (int tile = 0; tile < NT; ++tile)
      for (int kp = 0; kp < KP; ++kp)
        for (int lane = 0; lane < 32; ++lane) {
          const int gid = lane >> 2, tig = lane & 3;
          const float* w = rowptr(r, tile, gid);
          uint32_t* o = d + ((((size_t)r * NT + tile) * KP + kp) * 32 + lane) * 4;
          for (int q = 0; q < 4; ++q) {
            const int k = (2 * kp + (q >> 1)) * 16 + tig * 2 + (q & 1) * 8;
            o[q] = w ? (bf16_bits(w[k]) | (bf16_bits(w[k + 1]) << 16)) : 0u;
          }
        }
  return off;
}

// bf16 copy of a packed fp32 [N][K] matrix that already lives in the arena (2 values per float slot)
static size_t pack_bf16_copy(ArenaBuilder& ab, size_t src_off, size_t n) {
  size_t off = ab.add(nullptr, (n + 1) / 2);
  const float* s = ab.at(src_off);
  uint16_t* d = reinterpret_cast<uint16_t*>(ab.at(off));
  for (size_t i = 0; i < n; ++i) d[i] = (uint16_t)eh_bits(s[i]);
  return off;
}

// bf16 [N][taps][64] copy (input channels zero-padded to 64) of a packed fp32 [N][taps][Cin] conv weight
static size_t pack_bf16_conv_padded(ArenaBuilder& ab, size_t src_off, int N, int taps, int Cin) {
  size_t n = (size_t)N * taps * 64;
  size_t off = ab.add(nullptr, n / 2);
  const float* s = ab.at(src_off);
  uint16_t* d = reinterpret_cast<uint16_t*>(ab.at(off));
  for (size_t row = 0; row < (size_t)N * taps; ++row)
    for (int ci = 0; ci < 64; ++ci) d[row * 64 + ci] = ci < Cin ? (uint16_t)eh_bits(s[row * Cin + ci]) : 0;
  return off;
}

// B fragments of a 24 -> 24 3x3 convolution for conv3x3_c24_mma_kernel: k = tap * 24 + channel (216, zero-padded to
// 224), [k-step s][n-tile nt][lane] -> {b0 = W[n][16s + 2tig, +1], b1 = W[n][16s + 8 + 2tig, +1]}, n = 8 nt + gid.
static size_t pack_frag_conv24(ArenaBuilder& ab, size_t w_off) {
  const int K = 216;
  size_t off = ab.add(nullptr, (size_t)14 * 3 * 32 * 2);
  const float* w = ab.at(w_off);  // [24][216]
  uint32_t* d = reinterpret_cast<uint32_t*>(ab.at(off));
  for (int s = 0; s < 14; ++s)
    for (int nt = 0; nt < 3; ++nt)
      for (int lane = 0; lane < 32; ++lane) {
        const int gid = lane >> 2, tig = lane & 3, n = 8 * nt + gid;
        for (int q = 0; q < 2; ++q) {
          const int k = 16 * s + 8 * q + 2 * tig;
          const uint32_t lo = k < K ? eh_bits(w[(size_t)n * K + k]) : 0u, hi = k + 1 < K ? eh_bits(w[(size_t)n * K + k + 1]) : 0u;
          d[((size_t)(s * 3 + nt) * 32 + lane) * 2 + q] = lo | (hi << 16);
        }
      }
  return off;
}

static void pack_encoder_layers_bf16(frx_handle* h, ArenaBuilder& ab) {
  const size_t C = h->cfg.enc_hidden, F = h->cfg.enc_filter;
  for (EncLayerW& L : h->enc) {
    L.wb_qkv = pack_bf16_copy(ab, L.w_qkv, 3 * C * C);
    L.wb_o = pack_bf16_copy(ab, L.w_o, C * C);
    L.wb_c0 = pack_bf16_copy(ab, L.w_c0, F * C);
    L.wb_c1 = pack_bf16_copy(ab, L.w_c1, C * F);
  }
}

static void pack_encoder_bf16(frx_handle* h, ArenaBuilder& ab) {
  const frx_config& c = h->cfg;
  for (BlockW& b : h->blocks) {
    if (b.kind <= 1 && b.cin <= 64)
      b.wb_a_pad = pack_bf16_conv_padded(ab, b.w_a, b.kind == 0 ? b.cout : b.mid, b.k * b.k, b.cin);
    if (b.kind == 0) b.wb_a = pack_bf16_copy(ab, b.w_a, (size_t)b.cout * b.k * b.k * b.cin);
    if (b.kind == 0 && b.cin == 24 && b.cout == 24 && b.k == 3 && b.stride == 1) b.w_frag24 = pack_frag_conv24(ab, b.w_a);
    else if (b.kind == 1) {
      b.wb_a = pack_bf16_copy(ab, b.w_a, (size_t)b.mid * b.k * b.k * b.cin);
      b.wb_b = pack_bf16_copy(ab, b.w_b, (size_t)b.cout * b.mid);
    } else {
      b.wb_a = pack_bf16_copy(ab, b.w_a, (size_t)b.mid * b.cin);
      b.wb_b = pack_bf16_copy(ab, b.w_b, (size_t)b.cout * b.mid);
    }
  }
  h->last_wb = pack_bf16_copy(ab, h->last_w, (size_t)c.enc_hidden * 256);
  pack_encoder_layers_bf16(h, ab);
}

static int pack_decoder_bf16(frx_handle* h, ArenaBuilder& ab) {
  const frx_config& c = h->cfg;
  const int D = c.dec_hidden, F = c.dec_filter, V = c.num_classes, L = c.dec_layers;
  // the persistent cluster kernel exists for two geometries: EfficientSATRN (256 / 8 heads / 1024) and LiteSATRN
  // (128 / 4 heads / 512); one CTA per 32-wide head, 32 columns of D and 128 of F per CTA
  const bool geo = (D == 256 && F == 1024 && c.dec_heads == 8) || (D == 128 && F == 512 && c.dec_heads == 4) ||
                   (D == 512 && F == 512 && c.dec_heads == 8);   // SwinTRN decoder: 64-wide heads, one per CTA
  h->dec_cluster_ok = geo && L <= 4 && V <= 256;
  if (!h->dec_cluster_ok) return 0;  // e.g. SwinTRN (512 / 512 / 4 layers): the greedy loop stays on the fp32 step kernels
  auto W = [&](int l, const char* name) -> const float* {
    return find(h, "decoder.attention_layers." + std::to_string(l) + "." + name + ".weight")->f.data();
  };
  const float* gen = find(h, "decoder.generator.weight")->f.data();
  // row-major bf16 copies for the teacher-forced path (tcgen05 GEMMs want [N][K])
  h->gen_wb = pack_bf16_copy(ab, h->gen_w, (size_t)V * D);
  for (int l = 0; l < L; ++l) {
    DecLayerW& Wl = h->dec[l];
    Wl.wb_o = pack_bf16_copy(ab, Wl.w_o, (size_t)D * D);
    Wl.wb_q2 = pack_bf16_copy(ab, Wl.w_q2, (size_t)D * D);
    Wl.wb_o2 = pack_bf16_copy(ab, Wl.w_o2, (size_t)D * D);
    Wl.wb_f0 = pack_bf16_copy(ab, Wl.w_f0, (size_t)F * D);
    Wl.wb_f1 = pack_bf16_copy(ab, Wl.w_f1, (size_t)D * F);
    Wl.wb_sqkv = pack_bf16_copy(ab, Wl.w_sqkv, (size_t)3 * D * D);
  }
  // fragment packing for a cluster of CL CTAs; CTA r owns SW = D / CL columns of D (its heads) and FS = F / CL of the
  // FFN hidden row.  The 256-wide decoder is packed twice: one head per CTA (clusters of 8) and two (clusters of 4).
  auto pack_geometry = [&](int CL, std::vector<DecPackW>& dp, size_t& first) {
    const int SW = D / CL, FS = F / CL, NTS = SW / 8, NTE = FS / 8, NG = 256 / CL / 8;
    dp.assign(L, DecPackW{});
    first = pack_frag_stage(ab, CL, 3 * NTS, D, [&](int r, int tile, int gid) {
      const char* names[3] = {"self_attention_layer.q_linear", "self_attention_layer.k_linear", "self_attention_layer.v_linear"};
      return W(0, names[tile / NTS]) + (size_t)(r * SW + (tile % NTS) * 8 + gid) * D;
    });
    for (int l = 0; l < L; ++l) {
      DecPackW& P = dp[l];
      auto square = [&](const char* name, int K) {
        const float* w = W(l, name);
        return pack_frag_stage(ab, CL, NTS, K, [=](int r, int tile, int gid) { return w + (size_t)(r * SW + tile * 8 + gid) * K; });
      };
      P.w_o = square("self_attention_layer.out_linear", D);
      P.w_q2 = square("attention_layer.q_linear", D);
      P.w_o2 = square("attention_layer.out_linear", D);
      P.w_f1 = square("feedforward_layer.linear1", F);
      const float* f0 = W(l, "feedforward_layer.linear0");
      P.w_f0 = pack_frag_stage(ab, CL, NTE, D, [=](int r, int tile, int gid) {  // CTA r: hidden units [FS r, FS r + FS)
        return f0 + (size_t)(r * FS + tile * 8 + gid) * D;
      });
      const float* wk = W(l, "self_attention_layer.k_linear");
      const float* wv = W(l, "self_attention_layer.v_linear");
      if (l + 1 < L) {
        const float* nq = W(l + 1, "self_attention_layer.q_linear");
        const float* nk = W(l + 1, "self_attention_layer.k_linear");
        const float* nv = W(l + 1, "self_attention_layer.v_linear");
        P.w_next = pack_frag_stage(ab, CL, 5 * NTS, D, [=](int r, int tile, int gid) {
          const float* segs[5] = {wk, wv, nq, nk, nv};
          return segs[tile / NTS] + (size_t)(r * SW + (tile % NTS) * 8 + gid) * D;
        });
      } else {
        P.w_next = pack_frag_stage(ab, CL, 2 * NTS + NG, D, [=](int r, int tile, int gid) -> const float* {
          if (tile < 2 * NTS) return (tile < NTS ? wk : wv) + (size_t)(r * SW + (tile % NTS) * 8 + gid) * D;
          int n = r * (256 / CL) + (tile - 2 * NTS) * 8 + gid;
          return n < V ? gen + (size_t)n * D : nullptr;
        });
      }
    }
  };
  pack_geometry(c.dec_heads, h->dpack, h->dpack_first);
  if (D == 256) pack_geometry(c.dec_heads / 2, h->dpack2, h->dpack2_first);
  return 0;
}

extern "C" int frx_finalize_weights(frx_handle* h) {
  if (!h) return 1;
  const frx_config& c = h->cfg;
  ON_DEVICE(c.device);
  int down = c.network == FRX_NET_LITE_SATRN ? 16 : 32;
  h->feat_h = c.height / down;
  h->feat_w = c.width / down;
  ArenaBuilder ab;
  const bool want_enc = h->opt_parts & 1, want_dec = h->opt_parts & 2;
  if (want_enc) {
    if (c.network == FRX_NET_SWIN) {
      if (pack_swin(h, ab)) return 1;
    } else {
      if (c.network == FRX_NET_EFFICIENT_SATRN) {
        if (pack_trunk_efficientnet(h, ab)) return 1;
      } else if (pack_trunk_lite(h, ab)) {
        return 1;
      }
      if (pack_encoder(h, ab)) return 1;
    }
  }
  if (want_dec && pack_decoder(h, ab)) return 1;
  if (want_dec && c.precision == FRX_PREC_BF16 && pack_decoder_bf16(h, ab)) return 1;
  if (c.precision == FRX_PREC_BF16) {
    if (want_enc && c.network == FRX_NET_EFFICIENT_SATRN) pack_encoder_bf16(h, ab);
    if (want_enc && c.network == FRX_NET_LITE_SATRN) {
      for (int i = 1; i < 4; ++i) h->lite[i].wb = pack_bf16_copy(ab, h->lite[i].w, (size_t)h->lite[i].cout * 9 * h->lite[i].cin);
      pack_encoder_layers_bf16(h, ab);
    }
    if (want_enc && c.network == FRX_NET_SWIN) {
      for (SwinBlockW& b : h->sw_blocks) {
        const size_t C = b.dim;
        b.qkv_wb = pack_bf16_copy(ab, b.qkv_w, 3 * C * C);
        b.proj_wb = pack_bf16_copy(ab, b.proj_w, C * C);
        b.fc1_wb = pack_bf16_copy(ab, b.fc1_w, 4 * C * C);
        b.fc2_wb = pack_bf16_copy(ab, b.fc2_w, 4 * C * C);
      }
      for (SwinMergeW& m : h->sw_merges) m.red_wb = pack_bf16_copy(ab, m.red_w, (size_t)8 * m.dim * m.dim);
    }
    if (want_dec) h->cross_wb = pack_bf16_copy(ab, h->w_cross, (size_t)c.dec_layers * 2 * c.dec_hidden * c.dec_src);
  }
  // upload (re-finalize re-uses the arena when the size is unchanged).  Work enqueued earlier on ANY stream (torch side
  // streams are non-blocking with respect to the legacy stream) may still be reading the old weights: drain the device
  // before they are overwritten or freed.
  size_t bytes = ab.host.size() * sizeof(float);
  if (h->arena) CK(cudaDeviceSynchronize());
  if (!h->arena || h->arena_bytes != bytes) {
    if (h->arena) {
      for (size_t i = 0; i < h->allocs.size(); ++i)
        if (h->allocs[i] == (void*)h->arena) { h->allocs.erase(h->allocs.begin() + i); break; }
      cudaFree(h->arena);
      h->device_bytes -= (int64_t)h->arena_bytes;
      h->arena = nullptr;
    }
    void* p;
    if (dev_alloc(h, &p, bytes)) return 1;
    h->arena = (float*)p;
    h->arena_bytes = bytes;
  }
  CK(cudaMemcpy(h->arena, ab.host.data(), bytes, cudaMemcpyHostToDevice));

  if (!h->ws_ready) {
    // ---- activation workspaces sized for max_batch ------------------------
    const size_t B = c.max_batch;
    size_t act_max = 0, mid_max = 0;
    if (c.network == FRX_NET_EFFICIENT_SATRN) {
      int H = (c.height - 3) / 2 + 1, W = (c.width - 3) / 2 + 1;
      act_max = (size_t)H * W * 24;
      for (const BlockW& b : h->blocks) {
        int OH, OW, pl;
        same_pad(H, b.k, b.stride, &OH, &pl);
        same_pad(W, b.k, b.stride, &OW, &pl);
        size_t mid = b.kind == 1 ? (size_t)OH * OW * b.mid : (b.kind == 2 ? (size_t)H * W * b.mid : 0);
        if (mid > mid_max) mid_max = mid;
        H = OH; W = OW;
        if ((size_t)H * W * b.cout > act_max) act_max = (size_t)H * W * b.cout;
      }
    } else {
      act_max = (size_t)c.height * c.width * (c.enc_hidden / 2);
      mid_max = act_max;
    }
    size_t S = (size_t)h->feat_h * h->feat_w, C = c.enc_hidden;
    size_t enc_act = S * 3 * C;
    if (enc_act > mid_max) mid_max = enc_act;
    if (S * C > act_max) act_max = S * C;
    void* p;
    if (want_enc && c.network == FRX_NET_SWIN) {
      const size_t tok = 96 * 96;  // per image: x [tok,128], LN copy, q|k|v [tok,384], MLP hidden [tok,512] (largest at stage 0)
      for (int i = 0; i < 2; ++i) { if (dev_alloc(h, &p, B * tok * 128 * 4)) return 1; h->sw_x[i] = (float*)p; }
      if (dev_alloc(h, &p, B * tok * 128 * 4)) return 1; h->sw_a = (float*)p;
      if (dev_alloc(h, &p, B * tok * 384 * 4)) return 1; h->sw_qkv = (float*)p;
      if (dev_alloc(h, &p, B * tok * 512 * 4)) return 1; h->sw_hid = (float*)p;
      if (c.precision == FRX_PREC_BF16) {
        if (dev_alloc(h, &p, B * tok * 128 * 2)) return 1; h->sw_ab = p;
        if (dev_alloc(h, &p, B * tok * 512 * 2)) return 1; h->sw_hidb = p;
      }
    } else if (want_enc) {
      for (int i = 0; i < 2; ++i) { if (dev_alloc(h, &p, B * act_max * 4)) return 1; h->act[i] = (float*)p; }
      for (int i = 0; i < 2; ++i) { if (dev_alloc(h, &p, B * mid_max * 4)) return 1; h->mid[i] = (float*)p; }
      if (dev_alloc(h, &p, B * 2048 * 4 * 2)) return 1;  // SE means + gates
      h->gate = (float*)p;
    }
    // ---- decoder state ----------------------------------------------------
    const size_t D = c.dec_hidden, F = c.dec_filter, L = c.dec_layers, T = c.max_steps, V = c.num_classes;
    if (want_dec) {
    if (dev_alloc(h, &p, L * B * T * D * 4)) return 1; h->kself = (float*)p;
    if (dev_alloc(h, &p, L * B * T * D * 4)) return 1; h->vself = (float*)p;
    if (dev_alloc(h, &p, B * S * L * 2 * D * 4)) return 1; h->cross = (float*)p;
    float** small[] = {&h->dx, &h->datt, &h->dpre1, &h->dpre2, &h->du, &h->dw, &h->dq2};
    for (float** q : small) { if (dev_alloc(h, &p, B * D * 4)) return 1; *q = (float*)p; }
    if (dev_alloc(h, &p, B * 3 * D * 4)) return 1; h->dqkv = (float*)p;
    if (dev_alloc(h, &p, B * F * 4)) return 1; h->dff = (float*)p;
    if (dev_alloc(h, &p, B * T * V * 4)) return 1; h->logits_int = (float*)p;
    if (dev_alloc(h, &p, B * T * 8)) return 1; h->tokens_int = (long long*)p;
    if (dev_alloc(h, &p, B * T * 8)) return 1; h->forced_int = (long long*)p;
    if (dev_alloc(h, &p, B * 4)) return 1; h->cur_tok = (int*)p;
    if (dev_alloc(h, &p, 16)) return 1; h->eos_work = (int*)p;
    if (c.precision == FRX_PREC_BF16) {
      // self caches: [L][B][H][T][hd] by image, or [L][slots][H][T][hd] by cluster row in the stop-at-<EOS> decode,
      // whose slots = clusters * 8 round the batch up to a multiple of 8
      const size_t B8 = (B + DEC_IMG - 1) / DEC_IMG * DEC_IMG;
      if (dev_alloc(h, &p, L * B8 * T * D * 2)) return 1; h->kself_bf = p;
      if (dev_alloc(h, &p, L * B8 * T * D * 2)) return 1; h->vself_bf = p;
      if (dev_alloc(h, &p, L * B * S * D * 2)) return 1; h->kcross_bf = p;
      if (dev_alloc(h, &p, L * B * S * D * 2)) return 1; h->vcross_bf = p;
      if (dev_alloc(h, &p, B * S * (size_t)c.dec_src * 2)) return 1; h->mem_bf = p;
    }
    }
    if (dev_alloc(h, &p, B * S * C * 4)) return 1; h->memory_int = (float*)p;
    if (dev_alloc(h, &p, (size_t)c.in_ch * c.height * c.width * B * 4)) return 1; h->images_int = (float*)p;
    for (int i = 0; i < 5; ++i) CK(cudaEventCreate(&h->ev[i]));
    h->ws_ready = true;
  }
  // graphs bake arena pointers: drop them when weights are re-packed
  for (auto& kv : h->graphs) cudaGraphExecDestroy(kv.second.exec);
  h->graphs.clear();
  h->finalized = true;
  return 0;
}

// ---------------------------------------------------------------------------
// encoder
// ---------------------------------------------------------------------------
static int tap(frx_handle* h, const std::string& name, const float* src, int B, int H, int W, int C,
               cudaStream_t st) {
  if (!h->opt_taps) return 0;
  Tap& t = h->taps[name];
  size_t n = (size_t)B * H * W * C;
  if (t.capacity < n) {
    if (t.data) cudaFree(t.data);
    CK(cudaMalloc((void**)&t.data, n * 4));
    t.capacity = n;
  }
  t.shape[0] = B; t.shape[1] = H; t.shape[2] = W; t.shape[3] = C;
  CK(cudaMemcpyAsync(t.data, src, n * 4, cudaMemcpyDeviceToDevice, st));
  return 0;
}

extern "C" int frx_read_tap(frx_handle* h, const char* name, float* out, int64_t capacity, int64_t* count,
                            int32_t* shape4, void* stream) {
  if (!h || !name) return 1;
  auto it = h->taps.find(name);
  if (it == h->taps.end()) return fail(h, "no tap named '%s' (enable with frx_set_option(h,\"taps\",1))", name);
  const Tap& t = it->second;
  int64_t n = (int64_t)t.shape[0] * t.shape[1] * t.shape[2] * t.shape[3];
  if (count) *count = n;
  if (shape4) for (int i = 0; i < 4; ++i) shape4[i] = t.shape[i];
  if (out) {
    if (capacity < n) return fail(h, "tap '%s' needs %lld floats", name, (long long)n);
    CK(cudaMemcpyAsync(out, t.data, n * 4, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
  }
  return 0;
}

static int tap_bf16(frx_handle* h, const std::string& name, const void* src, int B, int H, int W, int C, cudaStream_t st) {
  if (!h->opt_taps) return 0;
  Tap& t = h->taps[name];
  size_t n = (size_t)B * H * W * C;
  if (t.capacity < n) {
    if (t.data) cudaFree(t.data);
    CK(cudaMalloc((void**)&t.data, n * 4));
    t.capacity = n;
  }
  t.shape[0] = B; t.shape[1] = H; t.shape[2] = W; t.shape[3] = C;
  launch_h16_to_f32((const eh_t*)src, t.data, (long long)n, st);
  CKL();
  return 0;
}

static GemmP dense_gemm(const float* A, int M, int K, const float* W, int N, float* C, int ldc) {
  GemmP g{};
  g.A = A; g.W = W; g.C = C; g.M = M; g.N = N; g.K = K; g.lda = K; g.ldc = ldc; g.conv = 0; g.rows_per_img = 1;
  return g;
}

static GemmP conv_gemm(const float* A, int B, int H, int W, int Cin, const float* Wt, int Cout, int k,
                       int stride, float* C, int* OH, int* OW) {
  GemmP g{};
  int pt, pl;
  same_pad(H, k, stride, OH, &pt);
  same_pad(W, k, stride, OW, &pl);
  g.A = A; g.W = Wt; g.C = C;
  g.M = B * (*OH) * (*OW); g.N = Cout; g.K = k * k * Cin; g.lda = 0; g.ldc = Cout;
  g.conv = 1; g.H = H; g.Wd = W; g.Cin = Cin; g.OH = *OH; g.OW = *OW; g.KH = k; g.KW = k;
  g.stride = stride; g.pad_t = pt; g.pad_l = pl; g.rows_per_img = 1;
  return g;
}

static int run_trunk_efficientnet(frx_handle* h, const float* images, int B, float** out, cudaStream_t st) {
  const frx_config& c = h->cfg;
  const float* A = h->arena;
  int H = (c.height - 3) / 2 + 1, W = (c.width - 3) / 2 + 1;
  float* x = h->act[0];
  float* y = h->act[1];
  launch_stem_conv(images, A + h->stem_w, A + h->stem_sc, A + h->stem_sh, x, B, c.in_ch, c.height, c.width, H, W, 24, st);
  CKL();
  if (tap(h, "stem", x, B, H, W, 24, st)) return 1;
  for (const BlockW& b : h->blocks) {
    int OH, OW;
    if (b.kind == 0) {
      GemmP g = conv_gemm(x, B, H, W, b.cin, A + b.w_a, b.cout, b.k, b.stride, y, &OH, &OW);
      g.scale = A + b.sc_a; g.shift = A + b.sh_a; g.act = ACT_SILU;
      if (b.residual) { g.res = x; g.ldr = b.cout; }
      launch_igemm_f32(g, st); CKL();
    } else if (b.kind == 1) {
      GemmP g = conv_gemm(x, B, H, W, b.cin, A + b.w_a, b.mid, b.k, b.stride, h->mid[0], &OH, &OW);
      g.scale = A + b.sc_a; g.shift = A + b.sh_a; g.act = ACT_SILU;
      launch_igemm_f32(g, st); CKL();
      GemmP g2 = dense_gemm(h->mid[0], B * OH * OW, b.mid, A + b.w_b, b.cout, y, b.cout);
      g2.scale = A + b.sc_b; g2.shift = A + b.sh_b; g2.act = ACT_NONE;
      if (b.residual) { g2.res = x; g2.ldr = b.cout; }
      launch_igemm_f32(g2, st); CKL();
    } else {
      GemmP g = dense_gemm(x, B * H * W, b.cin, A + b.w_a, b.mid, h->mid[0], b.mid);
      g.scale = A + b.sc_a; g.shift = A + b.sh_a; g.act = ACT_SILU;
      launch_igemm_f32(g, st); CKL();
      int pt, pl;
      same_pad(H, b.k, b.stride, &OH, &pt);
      same_pad(W, b.k, b.stride, &OW, &pl);
      DwP d{h->mid[0], A + b.w_dw, A + b.sc_dw, A + b.sh_dw, h->mid[1], B, H, W, b.mid, OH, OW, b.stride, pt, pl, ACT_SILU};
      launch_dwconv_f32(d, st); CKL();
      launch_se_gate_f32(h->mid[1], A + b.se_w1, A + b.se_b1, A + b.se_w2, A + b.se_b2, h->gate, B, OH * OW, b.mid, b.se_r, st);
      CKL();
      GemmP g2 = dense_gemm(h->mid[1], B * OH * OW, b.mid, A + b.w_b, b.cout, y, b.cout);
      g2.gate = h->gate; g2.rows_per_img = OH * OW;
      g2.scale = A + b.sc_b; g2.shift = A + b.sh_b; g2.act = ACT_NONE;
      if (b.residual) { g2.res = x; g2.ldr = b.cout; }
      launch_igemm_f32(g2, st); CKL();
    }
    H = OH; W = OW;
    float* t = x; x = y; y = t;
    if (tap(h, b.name, x, B, H, W, b.cout, st)) return 1;
  }
  GemmP g = dense_gemm(x, B * H * W, 256, A + h->last_w, c.enc_hidden, y, c.enc_hidden);
  g.scale = A + h->last_sc; g.shift = A + h->last_sh; g.act = ACT_SILU;
  launch_igemm_f32(g, st); CKL();
  if (H != h->feat_h || W != h->feat_w) return fail(h, "trunk output %dx%d != expected %dx%d", H, W, h->feat_h, h->feat_w);
  *out = y;
  return 0;
}

static TcGemmP tc_dense(const void* A, int M, int K, const float* arena, size_t w_off, int N, void* C, int out_f32) {
  TcGemmP g{};
  g.A = (const eh_t*)A; g.W = (const eh_t*)(arena + w_off); g.C = C;
  g.M = M; g.N = N; g.K = K; g.lda = K; g.ldw = K; g.ldc = N; g.out_f32 = out_f32;
  return g;
}

static TcGemmP tc_conv(const void* A, int B, int H, int W, int Cin, const float* arena, size_t w_off, int Cout, int k,
                       int stride, void* C, int* OH, int* OW) {
  TcGemmP g{};
  int pt, pl;
  same_pad(H, k, stride, OH, &pt);
  same_pad(W, k, stride, OW, &pl);
  g.A = (const eh_t*)A; g.W = (const eh_t*)(arena + w_off); g.C = C;
  g.M = B * (*OH) * (*OW); g.N = Cout; g.K = k * k * Cin; g.ldw = g.K; g.ldc = Cout;
  g.conv = 1; g.H = H; g.Wd = W; g.Cin = Cin; g.OH = *OH; g.OW = *OW; g.KW = k; g.stride = stride; g.pad_t = pt; g.pad_l = pl;
  return g;
}

#define TCL(g)                                                                                         \
  do {                                                                                                 \
    int rc__ = h->opt_tc_ws ? launch_tc_igemm_ws(g, h->num_sms, st) : launch_tc_igemm(g, st);          \
    if (rc__) return fail(h, "tcgen05 GEMM configuration failed: %s", cudaGetErrorString((cudaError_t)rc__)); \
    CKL();                                                                                             \
  } while (0)

// bf16 encoder: tcgen05 implicit GEMMs for every dense contraction, bf16 NHWC activations in the trunk,
// fp32 residual stream in the SATRN encoder layers.
// The SATRN encoder layers (EfficientSATRN.py:259-281) in 16-bit mode, shared by EfficientSATRN and LiteSATRN: LayerNorm
// (fp32 in, 16-bit out), q|k|v / out / conv0 / conv1 on the tcgen05 GEMM, attention on mma.sync, depthwise 3x3 on 16-bit
// NHWC.  xf: the positionally encoded tokens fp32 [M, C]; tf: a second fp32 [M, C] buffer (ping-pong for > 1 layer);
// m0 / m1: scratch (16-bit [M, max(C, F)] and fp32 [M, 3C]).
static int encoder_layers_16(frx_handle* h, float* tf, float* xf, eh_t* m0, eh_t* m1, int B, float* memory, cudaStream_t st) {
  typedef eh_t bf;
  const frx_config& c = h->cfg;
  const float* A = h->arena;
  const int fh = h->feat_h, fw = h->feat_w, S = fh * fw, C = c.enc_hidden, F = c.enc_filter, M = B * S;
  float* other = tf;
  for (int i = 0; i < c.enc_layers; ++i) {
    const EncLayerW& L = h->enc[i];
    launch_layernorm_bf16out(xf, nullptr, A + L.ln_g, A + L.ln_b, m0, M, C, 0, st); CKL();
    float* qkv = (float*)m1;
    TcGemmP g = tc_dense(m0, M, C, A, L.wb_qkv, 3 * C, qkv, 1);
    g.shift = A + L.b_qkv;
    TCL(g);
    if (!launch_enc_attn_mma_bf16(qkv, m0, B, S, C, c.enc_heads, st)) launch_enc_attn_bf16out(qkv, m0, B, S, C, c.enc_heads, st);
    CKL();
    float* proj = (float*)m1;
    TcGemmP go = tc_dense(m0, M, C, A, L.wb_o, C, proj, 1);
    go.shift = A + L.b_o;
    TCL(go);
    launch_layernorm_bf16out(proj, xf, A + L.ln_g, A + L.ln_b, m0, M, C, S, st); CKL();  // reinterpreted (:269) layout
    TcGemmP g0 = tc_dense(m0, M, C, A, L.wb_c0, F, m1, 0);
    g0.scale = A + L.sc_c0; g0.shift = A + L.sh_c0; g0.act = ACT_RELU;
    TCL(g0);
    launch_dwconv_bf16(m1, A + L.w_dw, A + L.sc_dw, A + L.sh_dw, m0, B, fh, fw, F, fh, fw, 1, 1, 1, ACT_RELU, st); CKL();
    float* dst = (i == c.enc_layers - 1) ? memory : other;
    TcGemmP g1 = tc_dense(m0, M, F, A, L.wb_c1, C, dst, 1);
    g1.scale = A + L.sc_c1; g1.shift = A + L.sh_c1; g1.act = ACT_RELU; g1.res = xf; g1.res_f32 = 1; g1.ldr = C;
    TCL(g1);
    if (tap(h, "enc_layer" + std::to_string(i), dst, B, fh, fw, C, st)) return 1;
    other = xf;
    xf = dst;
  }
  return 0;
}


static int encode_bf16(frx_handle* h, const float* images, int B, float* memory, cudaStream_t st) {
  const frx_config& c = h->cfg;
  const float* A = h->arena;
  typedef eh_t bf;
  int H = (c.height - 3) / 2 + 1, W = (c.width - 3) / 2 + 1;
  bf* x = (bf*)h->act[0];
  bf* y = (bf*)h->act[1];
  bf* m0 = (bf*)h->mid[0];
  bf* m1 = (bf*)h->mid[1];
  launch_stem_conv_bf16(images, A + h->stem_w, A + h->stem_sc, A + h->stem_sh, x, B, c.in_ch, c.height, c.width, H, W, 24, st);
  CKL();
  if (tap_bf16(h, "stem", x, B, H, W, 24, st)) return 1;
  for (const BlockW& b : h->blocks) {
    int OH, OW;
    if (b.kind == 0 && b.w_frag24 && h->opt_conv24) {
      OH = H; OW = W;  // 3x3, stride 1, "same"
      launch_conv3x3_c24_bf16(x, A + b.w_frag24, A + b.sc_a, A + b.sh_a, y, B, H, W, b.residual ? 1 : 0, st);
      CKL();
    } else if (b.kind == 0) {
      TcGemmP g = tc_conv(x, B, H, W, b.cin, A, b.wb_a, b.cout, b.k, b.stride, y, &OH, &OW);
      if (b.wb_a_pad && h->opt_tc_im2col) g.Wpad = (const eh_t*)(A + b.wb_a_pad);
      g.scale = A + b.sc_a; g.shift = A + b.sh_a; g.act = ACT_SILU;
      if (b.residual) { g.res = x; g.ldr = b.cout; }
      TCL(g);
    } else if (b.kind == 1) {
      TcGemmP g = tc_conv(x, B, H, W, b.cin, A, b.wb_a, b.mid, b.k, b.stride, m0, &OH, &OW);
      if (b.wb_a_pad && h->opt_tc_im2col) g.Wpad = (const eh_t*)(A + b.wb_a_pad);
      g.scale = A + b.sc_a; g.shift = A + b.sh_a; g.act = ACT_SILU;
      TCL(g);
      TcGemmP g2 = tc_dense(m0, B * OH * OW, b.mid, A, b.wb_b, b.cout, y, 0);
      g2.scale = A + b.sc_b; g2.shift = A + b.sh_b;
      if (b.residual) { g2.res = x; g2.ldr = b.cout; }
      TCL(g2);
    } else {
      TcGemmP g = tc_dense(x, B * H * W, b.cin, A, b.wb_a, b.mid, m0, 0);
      g.scale = A + b.sc_a; g.shift = A + b.sh_a; g.act = ACT_SILU;
      TCL(g);
      int pt, pl;
      same_pad(H, b.k, b.stride, &OH, &pt);
      same_pad(W, b.k, b.stride, &OW, &pl);
      launch_mbconv_dw_se_bf16(m0, A + b.w_dw, A + b.sc_dw, A + b.sh_dw, m1, h->gate, h->gate + (size_t)B * 2048,
                               A + b.se_w1, A + b.se_b1, A + b.se_w2t, A + b.se_b2, B, H, W, b.mid, OH, OW, b.stride, pt, pl,
                               b.se_r, st);
      CKL(); h->launches += 2;
      TcGemmP g2 = tc_dense(m1, B * OH * OW, b.mid, A, b.wb_b, b.cout, y, 0);
      g2.scale = A + b.sc_b; g2.shift = A + b.sh_b;
      if (b.residual) { g2.res = x; g2.ldr = b.cout; }
      TCL(g2);
    }
    H = OH; W = OW;
    bf* t = x; x = y; y = t;
    if (tap_bf16(h, b.name, x, B, H, W, b.cout, st)) return 1;
  }
  if (H != h->feat_h || W != h->feat_w) return fail(h, "trunk output %dx%d != expected %dx%d", H, W, h->feat_h, h->feat_w);
  const int fh = h->feat_h, fw = h->feat_w, S = fh * fw, C = c.enc_hidden, F = c.enc_filter, M = B * S;
  float* tf = (float*)y;  // conv_last output, fp32 [M, C]
  {
    TcGemmP g = tc_dense(x, M, 256, A, h->last_wb, C, tf, 1);
    g.scale = A + h->last_sc; g.shift = A + h->last_sh; g.act = ACT_SILU;
    TCL(g);
  }
  if (tap(h, "trunk", tf, B, fh, fw, C, st)) return 1;
  float* xf = (float*)x;
  launch_pe2d_f32(tf, A + h->pe_w0, A + h->pe_b0, A + h->pe_w1, A + h->pe_b1, A + h->pe_h, A + h->pe_w, xf, B, fh, fw, C, st);
  CKL();
  if (tap(h, "pe2d", xf, B, fh, fw, C, st)) return 1;
  return encoder_layers_16(h, tf, xf, m0, m1, B, memory, st);
}

// SwinTransformer.forward_features (SWIN.py:725-736) -> memory [B, 144, 1024]
static int encode_swin(frx_handle* h, const float* images, int B, float* memory, cudaStream_t st) {
  const float* A = h->arena;
  float* x = h->sw_x[0];
  float* y = h->sw_x[1];
  launch_swin_patch_embed(images, A + h->sw_pe_w, A + h->sw_pe_b, A + h->sw_pe_g, A + h->sw_pe_beta, A + h->sw_ape, x, B, 384,
                          96, 128, st);
  CKL();
  if (tap(h, "embed", x, B, 96, 96, 128, st)) return 1;
  size_t bi = 0;
  const int depths[4] = {2, 2, 18, 2};
  for (int i = 0; i < 4; ++i) {
    for (int j = 0; j < depths[i]; ++j, ++bi) {
      const SwinBlockW& b = h->sw_blocks[bi];
      const int M = B * b.res * b.res, C = b.dim;
      if (h->cfg.precision == FRX_PREC_BF16) {
        // bf16 mode: the four linear layers of the block on the tcgen05 GEMM (bf16 operands, fp32 accumulation);
        // residual stream, LayerNorm statistics and the window attention (softmax) stay fp32
        eh_t* ab16 = (eh_t*)h->sw_ab;
        launch_layernorm_bf16out(x, nullptr, A + b.n1_g, A + b.n1_b, ab16, M, C, 0, st); CKL();
        { TcGemmP g = tc_dense(ab16, M, C, A, b.qkv_wb, 3 * C, h->sw_qkv, 1); g.shift = A + b.qkv_b; TCL(g); }
        if (!launch_swin_window_attn_mma(h->sw_qkv, A + b.bias_table, ab16, B, b.res, C, b.heads, b.ws, b.shift, st)) {
          launch_swin_window_attn(h->sw_qkv, A + b.bias_table, h->sw_a, B, b.res, C, b.heads, b.ws, b.shift, st); CKL();
          launch_f32_to_h16(h->sw_a, ab16, (long long)M * C, st);
        }
        CKL();
        { TcGemmP g = tc_dense(ab16, M, C, A, b.proj_wb, C, y, 1); g.shift = A + b.proj_b; g.res = x; g.res_f32 = 1; g.ldr = C; TCL(g); }
        launch_layernorm_bf16out(y, nullptr, A + b.n2_g, A + b.n2_b, ab16, M, C, 0, st); CKL();
        { TcGemmP g = tc_dense(ab16, M, C, A, b.fc1_wb, 4 * C, h->sw_hidb, 0); g.shift = A + b.fc1_b; g.act = ACT_GELU; TCL(g); }
        { TcGemmP g = tc_dense(h->sw_hidb, M, 4 * C, A, b.fc2_wb, C, x, 1); g.shift = A + b.fc2_b; g.res = y; g.res_f32 = 1; g.ldr = C; TCL(g); }
        if (tap(h, "block" + std::to_string(i) + "." + std::to_string(j), x, B, b.res, b.res, C, st)) return 1;
        continue;
      }
      launch_layernorm_f32(x, nullptr, A + b.n1_g, A + b.n1_b, h->sw_a, M, C, 0, st); CKL();
      GemmP g = dense_gemm(h->sw_a, M, C, A + b.qkv_w, 3 * C, h->sw_qkv, 3 * C);
      g.shift = A + b.qkv_b;
      launch_igemm_f32(g, st); CKL();
      launch_swin_window_attn(h->sw_qkv, A + b.bias_table, h->sw_a, B, b.res, C, b.heads, b.ws, b.shift, st); CKL();
      GemmP gp = dense_gemm(h->sw_a, M, C, A + b.proj_w, C, y, C);   // y = x + proj(attn)
      gp.shift = A + b.proj_b; gp.res = x; gp.ldr = C;
      launch_igemm_f32(gp, st); CKL();
      launch_layernorm_f32(y, nullptr, A + b.n2_g, A + b.n2_b, h->sw_a, M, C, 0, st); CKL();
      GemmP g1 = dense_gemm(h->sw_a, M, C, A + b.fc1_w, 4 * C, h->sw_hid, 4 * C);
      g1.shift = A + b.fc1_b; g1.act = ACT_GELU;
      launch_igemm_f32(g1, st); CKL();
      GemmP g2 = dense_gemm(h->sw_hid, M, 4 * C, A + b.fc2_w, C, x, C);  // x = y + fc2(gelu(fc1(ln(y))))
      g2.shift = A + b.fc2_b; g2.res = y; g2.ldr = C;
      launch_igemm_f32(g2, st); CKL();
      if (tap(h, "block" + std::to_string(i) + "." + std::to_string(j), x, B, b.res, b.res, C, st)) return 1;
    }
    if (i < 3) {  // PatchMerging (:404-421)
      const SwinMergeW& m = h->sw_merges[i];
      const int M2 = B * (m.res / 2) * (m.res / 2);
      launch_swin_patch_merge(x, h->sw_hid, B, m.res, m.dim, st); CKL();
      if (h->cfg.precision == FRX_PREC_BF16) {
        launch_layernorm_bf16out(h->sw_hid, nullptr, A + m.n_g, A + m.n_b, (eh_t*)h->sw_hidb, M2, 4 * m.dim, 0, st); CKL();
        TcGemmP g = tc_dense(h->sw_hidb, M2, 4 * m.dim, A, m.red_wb, 2 * m.dim, x, 1);
        TCL(g);
        if (tap(h, "merge" + std::to_string(i), x, B, m.res / 2, m.res / 2, 2 * m.dim, st)) return 1;
        continue;
      }
      launch_layernorm_f32(h->sw_hid, nullptr, A + m.n_g, A + m.n_b, h->sw_qkv, M2, 4 * m.dim, 0, st); CKL();
      GemmP g = dense_gemm(h->sw_qkv, M2, 4 * m.dim, A + m.red_w, 2 * m.dim, x, 2 * m.dim);
      launch_igemm_f32(g, st); CKL();
      if (tap(h, "merge" + std::to_string(i), x, B, m.res / 2, m.res / 2, 2 * m.dim, st)) return 1;
    }
  }
  launch_layernorm_f32(x, nullptr, A + h->sw_norm_g, A + h->sw_norm_b, memory, B * 144, 1024, 0, st); CKL();
  return 0;
}

// LiteSATRN ShallowCNN (LiteSATRN.py:21-70): 4 x (conv3x3 p1 + BN + ReLU + maxpool2) -> H/16 x W/16 x hidden
static int run_trunk_lite(frx_handle* h, const float* images, int B, float** out, cudaStream_t st) {
  const frx_config& c = h->cfg;
  const float* A = h->arena;
  int H = c.height, W = c.width;
  float* x = h->act[0];
  float* y = h->act[1];
  if (c.precision == FRX_PREC_BF16 && !h->opt_enc_fp32 && h->lite[1].wb) {
    // bf16 mode: layer 0 fused with its max-pool (fp32 arithmetic on the single-channel image, bf16 NHWC out), layers
    // 1-3 as implicit GEMMs on the tcgen05 kernel (bf16 in / out, folded BN + ReLU in the epilogue), bf16 max-pools;
    // the last pool writes fp32 for the positional encoding / encoder layer that follow.
    typedef eh_t bf;
    bf* xb = (bf*)h->act[0];
    bf* yb = (bf*)h->act[1];
    const LiteConvW& L0 = h->lite[0];
    launch_lite_conv0_pool_bf16(images, A + L0.w, A + L0.sc, A + L0.sh, yb, B, L0.cin, H, W, L0.cout, st); CKL();
    H /= 2; W /= 2;
    for (int i = 1; i < 4; ++i) {
      const LiteConvW& L = h->lite[i];
      int OH, OW;
      TcGemmP g = tc_conv(yb, B, H, W, L.cin, A, L.wb, L.cout, 3, 1, xb, &OH, &OW);
      g.scale = A + L.sc; g.shift = A + L.sh; g.act = ACT_RELU;
      TCL(g);
      const bool last = i == 3;
      // the last pooled map goes to the second half of act[1] as fp32 (the bf16 input of this layer sits in the first half)
      float* f32_out = last ? h->act[1] + (size_t)B * (H / 2) * (W / 2) * L.cout : nullptr;
      launch_maxpool2_bf16(xb, yb, f32_out, B, H, W, L.cout, st); CKL();
      H /= 2; W /= 2;
      if (last) y = f32_out;
    }
    if (H != h->feat_h || W != h->feat_w) return fail(h, "trunk output %dx%d != expected %dx%d", H, W, h->feat_h, h->feat_w);
    if (tap(h, "lite_conv3", y, B, H, W, h->lite[3].cout, st)) return 1;
    *out = y;
    return 0;
  }
  for (int i = 0; i < 4; ++i) {
    const LiteConvW& L = h->lite[i];
    if (i == 0) {
      launch_direct_conv3x3(images, A + L.w, A + L.sc, A + L.sh, x, B, L.cin, H, W, H, W, L.cout, 1, 1, ACT_RELU, st);
      CKL();
    } else {
      int OH, OW;
      GemmP g = conv_gemm(y, B, H, W, L.cin, A + L.w, L.cout, 3, 1, x, &OH, &OW);
      g.scale = A + L.sc; g.shift = A + L.sh; g.act = ACT_RELU;
      launch_igemm_f32(g, st); CKL();
    }
    launch_maxpool2_f32(x, y, B, H, W, L.cout, st); CKL();
    H /= 2; W /= 2;
    if (tap(h, "lite_conv" + std::to_string(i), y, B, H, W, L.cout, st)) return 1;
  }
  if (H != h->feat_h || W != h->feat_w) return fail(h, "trunk output %dx%d != expected %dx%d", H, W, h->feat_h, h->feat_w);
  *out = y;
  return 0;
}

extern "C" int frx_encode(frx_handle* h, const float* images, int32_t B, float* memory, void* stream) {
  if (!h) return 1;
  if (!h->finalized) return fail(h, "frx_encode: weights not finalized");
  if (!(h->opt_parts & 1)) return fail(h, "frx_encode: handle was created without the encoder part");
  if (B <= 0 || B > h->cfg.max_batch) return fail(h, "frx_encode: batch %d outside (0, %d]", B, h->cfg.max_batch);
  const frx_config& c = h->cfg;
  cudaStream_t st = (cudaStream_t)stream;
  ON_DEVICE(c.device);
  if (c.network == FRX_NET_SWIN) return encode_swin(h, images, B, memory, st);
  if (c.precision == FRX_PREC_BF16 && !h->opt_enc_fp32 && c.network == FRX_NET_EFFICIENT_SATRN)
    return encode_bf16(h, images, B, memory, st);  // LiteSATRN in bf16 mode: fp32 ShallowCNN + encoder layer, bf16 decoder
  const float* A = h->arena;
  float* t = nullptr;
  if (c.network == FRX_NET_LITE_SATRN) {
    if (run_trunk_lite(h, images, B, &t, st)) return 1;
  } else if (run_trunk_efficientnet(h, images, B, &t, st)) {
    return 1;
  }
  const int fh = h->feat_h, fw = h->feat_w, S = fh * fw, C = c.enc_hidden, F = c.enc_filter;
  if (tap(h, "trunk", t, B, fh, fw, C, st)) return 1;
  float* x = (t == h->act[0]) ? h->act[1] : h->act[0];
  launch_pe2d_f32(t, A + h->pe_w0, A + h->pe_b0, A + h->pe_w1, A + h->pe_b1, A + h->pe_h, A + h->pe_w, x, B, fh, fw, C, st);
  CKL();
  if (tap(h, "pe2d", x, B, fh, fw, C, st)) return 1;
  if (c.network == FRX_NET_LITE_SATRN && c.precision == FRX_PREC_BF16 && !h->opt_enc_fp32 && h->enc[0].wb_qkv)
    return encoder_layers_16(h, t, x, (eh_t*)h->mid[0], (eh_t*)h->mid[1], B, memory, st);   // LiteSATRN, 16-bit mode
  float* other = t;
  const int M = B * S;
  for (int i = 0; i < c.enc_layers; ++i) {
    const EncLayerW& L = h->enc[i];
    float* ln = h->mid[0];          // [M,C]
    float* qkv = h->mid[1];         // [M,3C]
    launch_layernorm_f32(x, nullptr, A + L.ln_g, A + L.ln_b, ln, M, C, 0, st); CKL();
    GemmP g = dense_gemm(ln, M, C, A + L.w_qkv, 3 * C, qkv, 3 * C);
    g.shift = A + L.b_qkv;
    launch_igemm_f32(g, st); CKL();
    float* att = h->mid[0];         // ln no longer needed
    launch_enc_attn_f32(qkv, att, B, S, C, c.enc_heads, st); CKL();
    float* proj = h->mid[1];        // qkv no longer needed
    GemmP go = dense_gemm(att, M, C, A + L.w_o, C, proj, C);
    go.shift = A + L.b_o;
    launch_igemm_f32(go, st); CKL();
    float* scr = h->mid[0];         // LN(x + proj) stored in the reinterpreted (:269) layout
    launch_layernorm_f32(proj, x, A + L.ln_g, A + L.ln_b, scr, M, C, S, st); CKL();
    float* c0 = h->mid[1];
    GemmP g0 = dense_gemm(scr, M, C, A + L.w_c0, F, c0, F);
    g0.scale = A + L.sc_c0; g0.shift = A + L.sh_c0; g0.act = ACT_RELU;
    launch_igemm_f32(g0, st); CKL();
    float* dwo = h->mid[0];
    DwP d{c0, A + L.w_dw, A + L.sc_dw, A + L.sh_dw, dwo, B, fh, fw, F, fh, fw, 1, 1, 1, ACT_RELU};
    launch_dwconv_f32(d, st); CKL();
    float* dst = (i == c.enc_layers - 1) ? memory : other;
    GemmP g1 = dense_gemm(dwo, M, F, A + L.w_c1, C, dst, C);
    g1.scale = A + L.sc_c1; g1.shift = A + L.sh_c1; g1.act = ACT_RELU; g1.res = x; g1.ldr = C;
    launch_igemm_f32(g1, st); CKL();
    if (tap(h, "enc_layer" + std::to_string(i), dst, B, fh, fw, C, st)) return 1;
    other = x;
    x = dst;
  }
  return 0;
}

// ---------------------------------------------------------------------------
// decoder
// ---------------------------------------------------------------------------
static int run_cross_kv(frx_handle* h, const float* memory, int B, cudaStream_t st) {
  const frx_config& c = h->cfg;
  const int S = h->feat_h * h->feat_w;
  if (c.precision == FRX_PREC_BF16) {
    launch_f32_to_h16(memory, (eh_t*)h->mem_bf, (long long)B * S * c.dec_src, st); CKL();
    TcGemmP t = tc_dense(h->mem_bf, B * S, c.dec_src, h->arena, h->cross_wb, c.dec_layers * 2 * c.dec_hidden, h->cross, 1);
    t.shift = h->arena + h->b_cross;
    TCL(t);
    return 0;
  }
  GemmP g = dense_gemm(memory, B * S, c.dec_src, h->arena + h->w_cross, c.dec_layers * 2 * c.dec_hidden, h->cross,
                       c.dec_layers * 2 * c.dec_hidden);
  g.shift = h->arena + h->b_cross;
  launch_igemm_f32(g, st); CKL();
  return 0;
}

// One decoder step at position t for all B rows (SURVEY App. A.4).  The input
// row x must already be in h->dx.  Logits go to logits_dst[m*ld_logits + v].
struct StepRows {            // per-row (tree-structured) history for the best-first search; all nullptr = greedy
  const int* hist_len = nullptr;   // [B] number of cached rows attended
  const int* slot = nullptr;       // [B] cache row that receives this step's K/V
  const int* chain = nullptr;      // [B][T] cache rows of the ancestors
};

static int run_decode_step(frx_handle* h, int B, int t, float* logits_dst, long long ld_logits, cudaStream_t st,
                           const StepRows& rows = StepRows()) {
  const frx_config& c = h->cfg;
  const float* A = h->arena;
  const int D = c.dec_hidden, F = c.dec_filter, L = c.dec_layers, V = c.num_classes, T = c.max_steps;
  const int S = h->feat_h * h->feat_w, HD = D / c.dec_heads;
  const float temp = sqrtf((float)D);
  auto base_gemm = [&](const float* Ain, int K, const float* Wt, const float* bias, int N) {
    DecGemmP p{};
    p.A = Ain; p.Wt = Wt; p.bias = bias; p.M = B; p.N = N; p.K = K; p.lda = K; p.act = ACT_NONE;
    return p;
  };
  auto one_seg = [&](DecGemmP& p, float* dst, int ld) {
    p.nseg = 1;
    p.seg[0] = Seg{0, p.N, dst, ld, 0};
  };
  {  // layer 0 q|k|v of the embedded input
    DecGemmP p = base_gemm(h->dx, D, A + h->fused[0].wt, A + h->fused[0].b, 3 * D);
    one_seg(p, h->dqkv, 3 * D);
    launch_dec_gemm_f32(p, st); CKL();
  }
  for (int l = 0; l < L; ++l) {
    const DecLayerW& W = h->dec[l];
    float* kc = h->kself + (size_t)l * B * T * D;
    float* vc = h->vself + (size_t)l * B * T * D;
    {  // self attention over the t cached output rows + the current input row (:387-388)
      AttnP a{};
      a.q = h->dqkv; a.ldq = 3 * D; a.kcache = kc; a.vcache = vc; a.rows_per_img = T; a.D = D; a.n_hist = t;
      a.hist_len = rows.hist_len; a.chain = rows.chain; a.chain_stride = T;
      a.cur_k = h->dqkv + D; a.cur_v = h->dqkv + 2 * D; a.ld_cur = 3 * D; a.q_per_img = 1; a.temperature = temp;
      a.out = h->datt; a.ldo = D; a.M = B; a.heads = c.dec_heads;
      launch_dec_attn_f32(a, HD, st); CKL();
    }
    {  // pre1 = out_linear(a) + x
      DecGemmP p = base_gemm(h->datt, D, A + W.wt_o, A + W.b_o, D);
      p.res = h->dx; p.ldr = D;
      one_seg(p, h->dpre1, D);
      launch_dec_gemm_f32(p, st); CKL();
    }
    {  // u = LN(pre1); q2 = q_linear(u)
      DecGemmP p = base_gemm(h->dpre1, D, A + W.wt_q2, A + W.b_q2, D);
      p.ln_g = A + W.ln1_g; p.ln_b = A + W.ln1_b; p.a_norm_out = h->du;
      one_seg(p, h->dq2, D);
      launch_dec_gemm_f32(p, st); CKL();
    }
    {  // cross attention over the S memory tokens
      AttnP a{};
      a.q = h->dq2; a.ldq = D; a.kcache = h->cross + (size_t)l * 2 * D; a.vcache = h->cross + (size_t)l * 2 * D + D;
      a.rows_per_img = S; a.D = L * 2 * D; a.n_hist = S; a.q_per_img = 1; a.temperature = temp;
      a.out = h->datt; a.ldo = D; a.M = B; a.heads = c.dec_heads;
      launch_dec_attn_f32(a, HD, st); CKL();
    }
    {  // pre2 = out_linear(c) + u
      DecGemmP p = base_gemm(h->datt, D, A + W.wt_o2, A + W.b_o2, D);
      p.res = h->du; p.ldr = D;
      one_seg(p, h->dpre2, D);
      launch_dec_gemm_f32(p, st); CKL();
    }
    {  // w = LN(pre2); ff = relu(linear0(w))
      DecGemmP p = base_gemm(h->dpre2, D, A + W.wt_f0, A + W.b_f0, F);
      p.ln_g = A + W.ln2_g; p.ln_b = A + W.ln2_b; p.a_norm_out = h->dw; p.act = ACT_RELU;
      one_seg(p, h->dff, F);
      launch_dec_gemm_f32(p, st); CKL();
    }
    {  // pre1 = relu(linear1(ff)) + w      (:339-346 ReLU after both linears)
      DecGemmP p = base_gemm(h->dff, F, A + W.wt_f1, A + W.b_f1, D);
      p.act = ACT_RELU; p.res = h->dw; p.ldr = D;
      one_seg(p, h->dpre1, D);
      launch_dec_gemm_f32(p, st); CKL();
    }
    {  // y = LN(pre1) -> x ; K/V rows of y into the cache ; next layer's q|k|v or the logits
      const FusedW& Fw = h->fused[l + 1];
      DecGemmP p = base_gemm(h->dpre1, D, A + Fw.wt, A + Fw.b, Fw.N);
      p.ln_g = A + W.ln3_g; p.ln_b = A + W.ln3_b; p.a_norm_out = h->dx;
      p.nseg = 3;
      if (rows.slot) {
        p.row_slot = rows.slot;
        p.seg[0] = Seg{0, D, kc, (long long)T * D, D};
        p.seg[1] = Seg{D, 2 * D, vc, (long long)T * D, D};
      } else {
        p.seg[0] = Seg{0, D, kc + (size_t)t * D, (long long)T * D, 0};
        p.seg[1] = Seg{D, 2 * D, vc + (size_t)t * D, (long long)T * D, 0};
      }
      if (l + 1 < L) p.seg[2] = Seg{2 * D, 5 * D, h->dqkv, 3 * D, 0};
      else p.seg[2] = Seg{2 * D, 2 * D + V, logits_dst, ld_logits, 0};
      launch_dec_gemm_f32(p, st); CKL();
    }
  }
  return 0;
}

// mode 0: greedy, 1: forced tokens, 2: DecodingManager (the logits rows become masked softmax rows, :553-555)
static int run_greedy_loop(frx_handle* h, int B, int steps, int mode, cudaStream_t st) {
  const frx_config& c = h->cfg;
  const float* A = h->arena;
  const int D = c.dec_hidden, V = c.num_classes;
  const float scale = sqrtf((float)D);
  launch_dec_embed_f32(nullptr, nullptr, c.sos_id, A + h->emb, A + h->pe1d, 0, nullptr, 0, scale, h->dx, B, D, st);
  CKL();
  const SiftIds sids{h->sift_ids[0], h->sift_ids[1], h->sift_ids[2], h->sift_ids[3], h->sift_ids[4], h->sift_ids[5]};
  if (mode == 2) { launch_sift_state_init(h->sift_state, B, sids.sos, st); CKL(); }  // manager.reset (:536-537)
  for (int t = 0; t < steps; ++t) {
    float* lg = h->logits_int + (size_t)t * V;
    if (run_decode_step(h, B, t, lg, (long long)steps * V, st)) return 1;
    const float* pe_next = (t + 1 < steps) ? A + h->pe1d + (size_t)(t + 1) * D : nullptr;
    if (mode == 2)
      launch_dec_sift_embed(lg, (long long)steps * V, V, h->tokens_int + t, steps, h->sift_state, h->sift_flags,
                            h->sift_limit, sids, h->cur_tok, A + h->emb, pe_next, scale, h->dx, B, D, st);
    else
      launch_dec_argmax_embed(lg, (long long)steps * V, V, h->tokens_int + t, steps,
                              mode == 1 ? h->forced_int + t : nullptr, steps, h->cur_tok, A + h->emb, pe_next, scale,
                              h->dx, B, D, st);
    CKL();
  }
  return 0;
}

// "step mode" of the cluster kernel: continue per-image histories instead of decoding from <SOS> (DecClusterP)
struct ClusterStep {
  const int* hist_len = nullptr;
  const int* chain = nullptr;
  const int* slot = nullptr;
  const int* tok32 = nullptr;
  const long long* tok64 = nullptr;
};

static int cross_kv_to_bf16(frx_handle* h, int B, cudaStream_t st) {
  const frx_config& c = h->cfg;
  launch_cross_to_bf16(h->cross, (__nv_bfloat16*)h->kcross_bf, (__nv_bfloat16*)h->vcross_bf, B, h->feat_h * h->feat_w, c.dec_layers,
                       c.dec_hidden, c.dec_hidden / c.dec_heads, st);
  CKL();
  return 0;
}

// eos_lengths != nullptr: the stop-at-<EOS> instantiation (one launch for the whole batch, rows refilled from a work
// counter); it writes logits / tokens up to each image's length only.
static int decode_greedy_bf16(frx_handle* h, int B, int steps, float* logits, long long* tokens,
                              const long long* forced, cudaStream_t st, const ClusterStep* sm = nullptr, bool managed = false,
                              int* eos_lengths = nullptr) {
  const frx_config& c = h->cfg;
  const float* A = h->arena;
  const int S = h->feat_h * h->feat_w, L = c.dec_layers, D = c.dec_hidden;
  if (steps > DEC_TMAX) return fail(h, "bf16 decode kernel supports at most %d steps", DEC_TMAX);
  if (!sm && cross_kv_to_bf16(h, B, st)) return 1;      // step mode: converted once by the caller
  DecClusterP p{};
  if (sm) { p.hist_len = sm->hist_len; p.chain = sm->chain; p.slot = sm->slot; p.first_tok32 = sm->tok32; p.first_tok64 = sm->tok64; }
  if (managed) {   // DecodingManager: the rule tables go to the kernel's pick stage
    p.sift_flags = h->sift_flags; p.sift_limit = h->sift_limit;
    p.sift_ids = SiftIds{h->sift_ids[0], h->sift_ids[1], h->sift_ids[2], h->sift_ids[3], h->sift_ids[4], h->sift_ids[5]};
  }
  p.B = B; p.steps = steps; p.T = c.max_steps; p.L = L; p.V = c.num_classes; p.S = S; p.sos = c.sos_id;
  // 256-wide decoder: with one head per CTA (clusters of 8) only 15 clusters get their CTAs alone on an SM (an 8-CTA
  // cluster must sit inside one GPC); beyond that two CTAs share an SM and step in 67 us instead of 42.  Two heads per CTA
  // (clusters of 4 x 16 warps) keep every CTA alone on its SM up to 33 clusters; a cluster steps in ~57 us that way, so
  // batches of up to 15 clusters keep one head per CTA.  Option "dec_hpc" = 1 / 2 forces either.
  const int clusters = (B + DEC_IMG - 1) / DEC_IMG;
  const int want_hpc = h->opt_dec_hpc ? h->opt_dec_hpc : (clusters > 15 ? 2 : 1);
  const bool p2 = D == 256 && want_hpc == 2 && !h->dpack2.empty();
  const std::vector<DecPackW>& dpk = p2 ? h->dpack2 : h->dpack;
  p.w_first = reinterpret_cast<const uint4*>(A + (p2 ? h->dpack2_first : h->dpack_first));
  p.b_first = A + h->fused[0].b;
  for (int l = 0; l < L; ++l) {
    const DecPackW& P = dpk[l];
    const DecLayerW& W = h->dec[l];
    DecClusterLayer& Q = p.layer[l];
    Q.w_o = reinterpret_cast<const uint4*>(A + P.w_o);   Q.w_q2 = reinterpret_cast<const uint4*>(A + P.w_q2);
    Q.w_o2 = reinterpret_cast<const uint4*>(A + P.w_o2); Q.w_f0 = reinterpret_cast<const uint4*>(A + P.w_f0);
    Q.w_f1 = reinterpret_cast<const uint4*>(A + P.w_f1); Q.w_next = reinterpret_cast<const uint4*>(A + P.w_next);
    Q.b_o = A + W.b_o; Q.b_q2 = A + W.b_q2; Q.b_o2 = A + W.b_o2; Q.b_f0 = A + W.b_f0; Q.b_f1 = A + W.b_f1;
    Q.b_next = A + h->fused[l + 1].b;
    Q.ln1_g = A + W.ln1_g; Q.ln1_b = A + W.ln1_b; Q.ln2_g = A + W.ln2_g; Q.ln2_b = A + W.ln2_b;
    Q.ln3_g = A + W.ln3_g; Q.ln3_b = A + W.ln3_b;
  }
  p.emb = A + h->emb; p.pe = A + h->pe1d;
  p.kself = (__nv_bfloat16*)h->kself_bf; p.vself = (__nv_bfloat16*)h->vself_bf;
  p.kcross = (const __nv_bfloat16*)h->kcross_bf; p.vcross = (const __nv_bfloat16*)h->vcross_bf;
  p.logits = logits; p.tokens = tokens; p.forced = forced;
  p.prof = h->opt_prof ? h->prof : nullptr;
  if (p.prof) CK(cudaMemsetAsync(h->prof, 0, 16 * 8, st));
  if (eos_lengths) {
    p.lengths = eos_lengths; p.work = h->eos_work; p.eos = c.eos_id;
    CK(cudaMemsetAsync(h->eos_work, 0, sizeof(int), st));
  }
  if (h->opt_timing) CK(cudaEventRecord(h->ev[3], st));
  int rc = eos_lengths
               ? (D == 128 ? launch_dec_cluster_bf16_d128_eos(p, st)
                           : D == 512 ? launch_dec_cluster_bf16_d512_eos(p, st)
                                      : (p2 ? launch_dec_cluster_bf16_p2_eos(p, st) : launch_dec_cluster_bf16_eos(p, st)))
               : D == 128 ? launch_dec_cluster_bf16_d128(p, st)
                    : D == 512 ? launch_dec_cluster_bf16_d512(p, st) : (p2 ? launch_dec_cluster_bf16_p2(p, st) : launch_dec_cluster_bf16(p, st));
  if (rc) return fail(h, "decode cluster kernel configuration failed: %s", cudaGetErrorString((cudaError_t)rc));
  CKL();
  if (h->opt_timing) CK(cudaEventRecord(h->ev[4], st));
  h->timed_kernel = h->opt_timing;
  return 0;
}

// eos_lengths != nullptr: stop-at-<EOS> decode (frx_decode_greedy_eos).  The 16-bit cluster kernel stops each image at
// its <EOS>; the other paths decode all `steps` and apply the same contract afterwards (no time saved there).
static int decode_greedy_impl(frx_handle* h, const float* memory, int B, int steps, float* logits,
                              int64_t* tokens, const int64_t* forced, cudaStream_t st, bool managed = false,
                              int* eos_lengths = nullptr) {
  const frx_config& c = h->cfg;
  if (!h->finalized) return fail(h, "decode: weights not finalized");
  if (!(h->opt_parts & 2)) return fail(h, "decode: handle was created without the decoder part");
  if (B <= 0 || B > c.max_batch) return fail(h, "decode: batch %d outside (0, %d]", B, c.max_batch);
  if (steps <= 0 || steps > c.max_steps) return fail(h, "decode: steps %d outside (0, %d]", steps, c.max_steps);
  if (steps > 500) return fail(h, "decode: steps exceed the 1-D positional table (500)");
  ON_DEVICE(c.device);
  if (run_cross_kv(h, memory, B, st)) return 1;
  if (managed && !h->have_rules) return fail(h, "managed decode: frx_set_decoding_rules has not been called");
  if (managed && forced) return fail(h, "managed decode: forced tokens are not supported");
  const int mode = managed ? 2 : (forced ? 1 : 0);
  // bf16 mode: one persistent kernel that writes the caller's buffers directly.  Sequences longer than the kernel's
  // history capacity (the reference decodes up to the 500 rows of its 1-D positional table) take the step-kernel loop.
  if (c.precision == FRX_PREC_BF16 && h->dec_cluster_ok && steps <= DEC_TMAX && (!managed || h->opt_step16)) {
    long long* tok = (long long*)(tokens ? tokens : (int64_t*)h->tokens_int);
    if (decode_greedy_bf16(h, B, steps, logits, tok, (const long long*)forced, st, nullptr, managed, eos_lengths)) return 1;
    if (eos_lengths) { launch_eos_finalize(logits, tok, eos_lengths, nullptr, B, steps, c.num_classes, c.eos_id, c.pad_id, true, st); CKL(); }
    return 0;
  }
  if (forced) CK(cudaMemcpyAsync(h->forced_int, forced, (size_t)B * steps * 8, cudaMemcpyDeviceToDevice, st));
  if (h->opt_graphs) {
    GraphKey key{B, steps, mode};
    auto it = h->graphs.find(key);
    if (it == h->graphs.end()) {
      cudaStream_t cs;
      CK(cudaStreamCreateWithFlags(&cs, cudaStreamNonBlocking));
      int64_t before = h->launches;
      CK(cudaStreamBeginCapture(cs, cudaStreamCaptureModeThreadLocal));
      int rc = run_greedy_loop(h, B, steps, mode, cs);
      cudaGraph_t graph = nullptr;
      cudaError_t e = cudaStreamEndCapture(cs, &graph);
      cudaStreamDestroy(cs);
      if (rc) { if (graph) cudaGraphDestroy(graph); return 1; }
      if (e != cudaSuccess) return fail(h, "graph capture failed: %s", cudaGetErrorString(e));
      GraphEntry ge{};
      ge.nodes = h->launches - before;
      h->launches = before;
      e = cudaGraphInstantiate(&ge.exec, graph, 0);
      cudaGraphDestroy(graph);
      if (e != cudaSuccess) return fail(h, "graph instantiate failed: %s", cudaGetErrorString(e));
      // bounded cache: validation batches come in many target lengths, and a 231-step graph holds ~6 000 kernel nodes
      if (h->graphs.size() >= FRX_MAX_GRAPHS) {
        auto victim = h->graphs.begin();
        for (auto g = h->graphs.begin(); g != h->graphs.end(); ++g)
          if (g->second.last_use < victim->second.last_use) victim = g;
        CK(cudaStreamSynchronize(st));   // the evicted exec may still be running on this stream
        cudaGraphExecDestroy(victim->second.exec);
        h->graphs.erase(victim);
      }
      it = h->graphs.emplace(key, ge).first;
    }
    it->second.last_use = ++h->graph_clock;
    CK(cudaGraphLaunch(it->second.exec, st));
    h->launches += it->second.nodes;
  } else if (run_greedy_loop(h, B, steps, mode, st)) {
    return 1;
  }
  if (logits) CK(cudaMemcpyAsync(logits, h->logits_int, (size_t)B * steps * c.num_classes * 4, cudaMemcpyDeviceToDevice, st));
  if (tokens) CK(cudaMemcpyAsync(tokens, h->tokens_int, (size_t)B * steps * 8, cudaMemcpyDeviceToDevice, st));
  if (eos_lengths) {
    long long* tok = (long long*)(tokens ? tokens : (int64_t*)h->tokens_int);
    launch_eos_finalize(logits, tok, eos_lengths, forced ? (const long long*)forced : tok, B, steps, c.num_classes, c.eos_id,
                        c.pad_id, false, st);
    CKL();
  }
  return 0;
}

extern "C" int frx_decode_greedy(frx_handle* h, const float* memory, int32_t B, int32_t steps, float* logits,
                                 int64_t* tokens, const int64_t* forced, void* stream) {
  if (!h) return 1;
  return decode_greedy_impl(h, memory, B, steps, logits, tokens, forced, (cudaStream_t)stream);
}

extern "C" int frx_decode_greedy_eos(frx_handle* h, const float* memory, int32_t B, int32_t max_steps, float* logits,
                                     int64_t* tokens, int32_t* lengths, const int64_t* forced, int32_t managed, void* stream) {
  if (!h) return 1;
  if (!lengths) return fail(h, "decode_greedy_eos: lengths must not be NULL");
  return decode_greedy_impl(h, memory, B, max_steps, logits, tokens, forced, (cudaStream_t)stream, managed != 0, lengths);
}

extern "C" int frx_forward_greedy_eos(frx_handle* h, const float* images, int32_t B, int32_t max_steps, float* logits,
                                      int64_t* tokens, int32_t* lengths, int32_t managed, void* stream) {
  if (!h) return 1;
  if (frx_encode(h, images, B, h->memory_int, stream)) return 1;
  return frx_decode_greedy_eos(h, h->memory_int, B, max_steps, logits, tokens, lengths, nullptr, managed, stream);
}

// DecodingManager (postprocessing/postprocessing.py:182-405): upload the per-token rule tables.
extern "C" int frx_set_decoding_rules(frx_handle* h, const int32_t* flags, const int32_t* limit, int32_t num_classes,
                                      const int32_t* ids6) {
  if (!h) return 1;
  const frx_config& c = h->cfg;
  if (num_classes != c.num_classes) return fail(h, "decoding rules: %d classes, the model has %d", num_classes, c.num_classes);
  for (int i = 0; i < 6; ++i)
    if (ids6[i] < 0 || ids6[i] >= num_classes) return fail(h, "decoding rules: special token id %d out of range", ids6[i]);
  ON_DEVICE(c.device);
  if (!h->sift_flags) {
    void* p;
    if (dev_alloc(h, &p, (size_t)num_classes * 4)) return 1; h->sift_flags = (int*)p;
    if (dev_alloc(h, &p, (size_t)num_classes * 4)) return 1; h->sift_limit = (int*)p;
    if (dev_alloc(h, &p, (size_t)c.max_batch * sizeof(int4))) return 1; h->sift_state = (int4*)p;
  }
  CK(cudaMemcpy(h->sift_flags, flags, (size_t)num_classes * 4, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(h->sift_limit, limit, (size_t)num_classes * 4, cudaMemcpyHostToDevice));
  for (int i = 0; i < 6; ++i) h->sift_ids[i] = ids6[i];
  h->have_rules = true;
  for (auto it = h->graphs.begin(); it != h->graphs.end();) {  // captured graphs embed the special-token ids
    if (std::get<2>(it->first) == 2) { cudaGraphExecDestroy(it->second.exec); it = h->graphs.erase(it); }
    else ++it;
  }
  return 0;
}

// SATRNDecoder.forward inference branch with a DecodingManager attached (EfficientSATRN.py:536-564).
extern "C" int frx_decode_greedy_managed(frx_handle* h, const float* memory, int32_t B, int32_t steps, float* probs,
                                         int64_t* tokens, void* stream) {
  if (!h) return 1;
  return decode_greedy_impl(h, memory, B, steps, probs, tokens, nullptr, (cudaStream_t)stream, true);
}

extern "C" int frx_forward_greedy_managed(frx_handle* h, const float* images, int32_t B, int32_t steps, float* probs,
                                          int64_t* tokens, void* stream) {
  if (!h) return 1;
  if (frx_encode(h, images, B, h->memory_int, stream)) return 1;
  return decode_greedy_impl(h, h->memory_int, B, steps, probs, tokens, nullptr, (cudaStream_t)stream, true);
}

extern "C" int frx_forward_greedy(frx_handle* h, const float* images, int32_t B, int32_t steps, float* logits,
                                  int64_t* tokens, void* stream) {
  if (!h) return 1;
  cudaStream_t st = (cudaStream_t)stream;
  if (h->opt_timing) CK(cudaEventRecord(h->ev[0], st));
  if (frx_encode(h, images, B, h->memory_int, stream)) return 1;
  if (h->opt_timing) CK(cudaEventRecord(h->ev[1], st));
  if (decode_greedy_impl(h, h->memory_int, B, steps, logits, tokens, nullptr, st)) return 1;
  if (h->opt_timing) {
    CK(cudaEventRecord(h->ev[2], st));
    CK(cudaEventSynchronize(h->ev[2]));
    CK(cudaEventElapsedTime(&h->last_ms[0], h->ev[0], h->ev[1]));
    CK(cudaEventElapsedTime(&h->last_ms[1], h->ev[1], h->ev[2]));
    CK(cudaEventElapsedTime(&h->last_ms[2], h->ev[0], h->ev[2]));
    h->last_ms[3] = 0.f;
    if (h->timed_kernel) CK(cudaEventElapsedTime(&h->last_ms[3], h->ev[3], h->ev[4]));
  }
  return 0;
}

extern "C" int frx_forward_greedy_host(frx_handle* h, const float* images_host, int32_t B, int32_t steps,
                                       float* logits_host, int64_t* tokens_host, void* stream) {
  if (!h) return 1;
  if (!h->finalized) return fail(h, "forward: weights not finalized");
  const frx_config& c = h->cfg;
  if (B <= 0 || B > c.max_batch) return fail(h, "forward: batch %d outside (0, %d]", B, c.max_batch);
  cudaStream_t st = (cudaStream_t)stream;
  ON_DEVICE(c.device);
  size_t img_bytes = (size_t)B * c.in_ch * c.height * c.width * 4;
  CK(cudaMemcpyAsync(h->images_int, images_host, img_bytes, cudaMemcpyHostToDevice, st));
  if (frx_forward_greedy(h, h->images_int, B, steps,
                         (c.precision == FRX_PREC_BF16 && logits_host) ? h->logits_int : nullptr,
                         (c.precision == FRX_PREC_BF16) ? (int64_t*)h->tokens_int : nullptr, stream))
    return 1;
  if (tokens_host) CK(cudaMemcpyAsync(tokens_host, h->tokens_int, (size_t)B * steps * 8, cudaMemcpyDeviceToHost, st));
  if (logits_host) CK(cudaMemcpyAsync(logits_host, h->logits_int, (size_t)B * steps * c.num_classes * 4, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  return 0;
}

// 16-bit handles run single decoder steps (step_forward, ensembles, best-first search) on the cluster kernel too;
// option "step16" = 0 keeps them on the fp32 step kernels (the bit-faithful path the fp32 goldens pin).
static bool step16(const frx_handle* h) {
  return h->cfg.precision == FRX_PREC_BF16 && h->dec_cluster_ok && h->opt_step16 && h->cfg.max_steps <= DEC_TMAX;
}

// Pipelined host entry: batch i + 1's images travel host -> device and batch i - 1's tokens device -> host on their own
// streams while batch i computes on `stream`.  Two slots; a slot may be re-submitted after frx_forward_greedy_host_wait.
// The ENCODER of batch i + 1 also runs on its own stream: the persistent decode kernel of batch i occupies 128 of the 148
// SMs (one 512-thread CTA each) for ~15 ms with a quarter of its issue slots busy, so the next batch's encoder kernels
// start on the 20 idle SMs under it and finish at full width once it retires (encoder and decoder share no workspace:
// each slot has its own encoder-output buffer).
extern "C" int frx_forward_greedy_host_submit(frx_handle* h, const float* images_host, int32_t B, int32_t steps,
                                              int64_t* tokens_host, int32_t slot, void* stream) {
  if (!h) return 1;
  if (!h->finalized) return fail(h, "forward: weights not finalized");
  const frx_config& c = h->cfg;
  if (B <= 0 || B > c.max_batch) return fail(h, "forward: batch %d outside (0, %d]", B, c.max_batch);
  if (steps <= 0 || steps > c.max_steps) return fail(h, "forward: steps %d outside (0, %d]", steps, c.max_steps);
  if (slot < 0 || slot > 1 || !images_host || !tokens_host) return fail(h, "host_submit: slot must be 0 or 1 and both host buffers given");
  if (h->opt_timing) return fail(h, "host_submit: option 'timing' synchronises every call; switch it off for the pipelined entry");
  cudaStream_t st = (cudaStream_t)stream;
  ON_DEVICE(c.device);
  frx_handle::PipeSlot& sl = h->pipe[slot];
  if (sl.busy) return fail(h, "host_submit: slot %d is still in flight (call frx_forward_greedy_host_wait first)", slot);
  if (!h->pipe_h2d) {
    CK(cudaStreamCreateWithFlags(&h->pipe_h2d, cudaStreamNonBlocking));
    CK(cudaStreamCreateWithFlags(&h->pipe_d2h, cudaStreamNonBlocking));
    CK(cudaStreamCreateWithFlags(&h->pipe_enc, cudaStreamNonBlocking));
  }
  if (!sl.img) {
    void* p;
    if (dev_alloc(h, &p, (size_t)c.max_batch * c.in_ch * c.height * c.width * 4)) return 1; sl.img = (float*)p;
    if (dev_alloc(h, &p, (size_t)c.max_batch * c.max_steps * 8)) return 1; sl.tok = (long long*)p;
    if (dev_alloc(h, &p, (size_t)c.max_batch * h->feat_h * h->feat_w * c.enc_hidden * 4)) return 1; sl.mem = (float*)p;
    CK(cudaEventCreateWithFlags(&sl.h2d, cudaEventDisableTiming));
    CK(cudaEventCreateWithFlags(&sl.enc, cudaEventDisableTiming));
    CK(cudaEventCreateWithFlags(&sl.done, cudaEventDisableTiming));
    CK(cudaEventCreateWithFlags(&sl.d2h, cudaEventDisableTiming));
  }
  const size_t img_bytes = (size_t)B * c.in_ch * c.height * c.width * 4;
  CK(cudaMemcpyAsync(sl.img, images_host, img_bytes, cudaMemcpyDefault, h->pipe_h2d));   // host (pinned) or device source
  CK(cudaEventRecord(sl.h2d, h->pipe_h2d));
  const bool split = h->opt_pipe_enc && (h->opt_parts & 3) == 3;
  if (split) {
    // encoder on its own stream (its activations are private to it and calls are serialised on that stream)
    CK(cudaStreamWaitEvent(h->pipe_enc, sl.h2d, 0));
    if (frx_encode(h, sl.img, B, sl.mem, (void*)h->pipe_enc)) return 1;
    CK(cudaEventRecord(sl.enc, h->pipe_enc));
    CK(cudaStreamWaitEvent(st, sl.enc, 0));
    if (decode_greedy_impl(h, sl.mem, B, steps, nullptr, (int64_t*)sl.tok, nullptr, st)) return 1;
  } else {
    CK(cudaStreamWaitEvent(st, sl.h2d, 0));
    if (frx_forward_greedy(h, sl.img, B, steps, nullptr, (int64_t*)sl.tok, stream)) return 1;
  }
  CK(cudaEventRecord(sl.done, st));
  CK(cudaStreamWaitEvent(h->pipe_d2h, sl.done, 0));
  CK(cudaMemcpyAsync(tokens_host, sl.tok, (size_t)B * steps * 8, cudaMemcpyDefault, h->pipe_d2h));
  CK(cudaEventRecord(sl.d2h, h->pipe_d2h));
  sl.busy = true;
  return 0;
}

extern "C" int frx_forward_greedy_host_wait(frx_handle* h, int32_t slot) {
  if (!h) return 1;
  if (slot < 0 || slot > 1) return fail(h, "host_wait: slot must be 0 or 1");
  frx_handle::PipeSlot& sl = h->pipe[slot];
  if (!sl.busy) return 0;
  ON_DEVICE(h->cfg.device);
  CK(cudaEventSynchronize(sl.d2h));
  sl.busy = false;
  return 0;
}

extern "C" int frx_decode_begin(frx_handle* h, const float* memory, int32_t B, void* stream) {
  if (!h) return 1;
  if (!h->finalized) return fail(h, "decode_begin: weights not finalized");
  if (!(h->opt_parts & 2)) return fail(h, "decode_begin: handle was created without the decoder part");
  if (B <= 0 || B > h->cfg.max_batch) return fail(h, "decode_begin: batch %d outside (0, %d]", B, h->cfg.max_batch);
  ON_DEVICE(h->cfg.device);
  if (run_cross_kv(h, memory, B, (cudaStream_t)stream)) return 1;
  if (step16(h) && cross_kv_to_bf16(h, B, (cudaStream_t)stream)) return 1;
  h->step_idx = 0;
  h->step_batch = B;
  return 0;
}

extern "C" int frx_decode_step(frx_handle* h, const int64_t* target, float* logits, void* stream) {
  if (!h) return 1;
  if (h->step_batch <= 0) return fail(h, "decode_step: call frx_decode_begin first");
  if (h->step_idx >= h->cfg.max_steps) return fail(h, "decode_step: step %d exceeds max_steps %d", h->step_idx, h->cfg.max_steps);
  const frx_config& c = h->cfg;
  cudaStream_t st = (cudaStream_t)stream;
  ON_DEVICE(c.device);
  if (step16(h)) {
    // 16-bit handle: ONE launch of the cluster kernel in step mode (history length = step_idx for every image) instead
    // of the ~26 fp32 step kernels
    if (!h->step_hist) { void* q; if (dev_alloc(h, &q, (size_t)c.max_batch * 4)) return 1; h->step_hist = (int*)q; }
    launch_fill_i32(h->step_hist, h->step_idx, h->step_batch, st); CKL();
    ClusterStep sm;
    sm.hist_len = h->step_hist; sm.tok64 = (const long long*)target;
    if (decode_greedy_bf16(h, h->step_batch, 1, logits, nullptr, nullptr, st, &sm)) return 1;
    h->step_idx++;
    return 0;
  }
  launch_dec_embed_f32(nullptr, (const long long*)target, 0, h->arena + h->emb, h->arena + h->pe1d, h->step_idx, nullptr, 0,
                       sqrtf((float)c.dec_hidden), h->dx, h->step_batch, c.dec_hidden, st);
  CKL();
  if (run_decode_step(h, h->step_batch, h->step_idx, logits, c.num_classes, st)) return 1;
  h->step_idx++;
  return 0;
}

static int ws_alloc(frx_handle* h, void** p, size_t bytes) {
  if (*p) return 0;
  return dev_alloc(h, p, bytes);
}

// EfficientSATRN.beam_search (:708-867), topk = 1: all samples advance one expansion per round.
extern "C" int frx_beam_search(frx_handle* h, const float* memory, int32_t B, int32_t beam_width,
                               int32_t max_sequence, int64_t* tokens, void* stream) {
  if (!h) return 1;
  const frx_config& c = h->cfg;
  if (!h->finalized) return fail(h, "beam_search: weights not finalized");
  if (!(h->opt_parts & 2)) return fail(h, "beam_search: handle was created without the decoder part");
  if (B <= 0 || B > c.max_batch) return fail(h, "beam_search: batch %d outside (0, %d]", B, c.max_batch);
  if (beam_width < 1 || beam_width > 8) return fail(h, "beam_search: beam_width %d outside [1, 8]", beam_width);
  if (max_sequence < 2 || max_sequence > c.max_steps) return fail(h, "beam_search: max_sequence %d outside [2, %d]", max_sequence, c.max_steps);
  if (c.num_classes > 256) return fail(h, "beam_search: more than 256 classes not supported");
  cudaStream_t st = (cudaStream_t)stream;
  ON_DEVICE(c.device);
  const int T = c.max_steps, V = c.num_classes, D = c.dec_hidden;
  const size_t Bm = c.max_batch;
  const int cap = (T - 1) * 8 + 2;  // root + beam_width children per expansion
  BeamWs& w = h->beam;
  if (ws_alloc(h, (void**)&w.hscore, Bm * cap * 8) || ws_alloc(h, (void**)&w.hnode, Bm * cap * 4) ||
      ws_alloc(h, (void**)&w.nprev, Bm * cap * 4) || ws_alloc(h, (void**)&w.ntok, Bm * cap * 4) ||
      ws_alloc(h, (void**)&w.nlen, Bm * cap * 4) || ws_alloc(h, (void**)&w.nlogp, Bm * cap * 8) ||
      ws_alloc(h, (void**)&w.nkv, Bm * cap * 4) || ws_alloc(h, (void**)&w.chain, Bm * T * 4) ||
      ws_alloc(h, (void**)&w.small, Bm * 12 * 4 + 64) || ws_alloc(h, (void**)&w.logits, Bm * V * 4))
    return 1;
  if (!w.host_flag) CK(cudaMallocHost((void**)&w.host_flag, sizeof(int)));
  BeamP p{};
  p.B = B; p.V = V; p.bw = beam_width; p.max_seq = max_sequence; p.T = T; p.cap = cap;
  p.sos = c.sos_id; p.eos = c.eos_id; p.pad = c.pad_id;
  p.hscore = w.hscore; p.hnode = w.hnode; p.nprev = w.nprev; p.ntok = w.ntok; p.nlen = w.nlen; p.nlogp = w.nlogp;
  p.nkv = w.nkv; p.chain = w.chain;
  int* s = w.small;
  p.hsize = s; p.ncount = s + Bm; p.num_steps = s + 2 * Bm; p.done = s + 3 * Bm; p.endnode = s + 4 * Bm;
  p.nexp = s + 5 * Bm; p.cur_node = s + 6 * Bm; p.cur_tok = s + 7 * Bm; p.pos = s + 8 * Bm; p.slot = s + 9 * Bm;
  p.active = s + 10 * Bm; p.n_active = s + 11 * Bm;
  p.logits = w.logits; p.out = (long long*)tokens;
  if (run_cross_kv(h, memory, B, st)) return 1;
  const bool s16 = step16(h);
  if (s16 && cross_kv_to_bf16(h, B, st)) return 1;
  launch_beam_init(p, st); CKL();
  StepRows rows;
  rows.hist_len = p.pos; rows.slot = p.slot; rows.chain = p.chain;
  const float scale = sqrtf((float)D);
  const int max_rounds = max_sequence + 1;
  for (int round = 0; round < max_rounds; ++round) {
    CK(cudaMemsetAsync(p.n_active, 0, sizeof(int), st));
    launch_beam_select(p, st); CKL();
    if (s16) {   // one cluster-kernel launch per round: history = the node's ancestor chain, K/V row = the node's slot
      ClusterStep sm;
      sm.hist_len = p.pos; sm.chain = p.chain; sm.slot = p.slot; sm.tok32 = p.cur_tok;
      if (decode_greedy_bf16(h, B, 1, w.logits, nullptr, nullptr, st, &sm)) return 1;
    } else {
      launch_dec_embed_f32(p.cur_tok, nullptr, 0, h->arena + h->emb, h->arena + h->pe1d, 0, p.pos, 0, scale, h->dx, B, D, st);
      CKL();
      if (run_decode_step(h, B, 0, w.logits, V, st, rows)) return 1;
    }
    launch_beam_push(p, st); CKL();
    if ((round & 7) == 7 || round == max_rounds - 1) {  // every 8 rounds: has every sample finished?
      CK(cudaMemcpyAsync(w.host_flag, p.n_active, sizeof(int), cudaMemcpyDeviceToHost, st));
      CK(cudaStreamSynchronize(st));
      if (*w.host_flag == 0) break;
    }
  }
  launch_beam_finish(p, st); CKL();
  return 0;
}

// SATRNDecoder.forward, teacher-forced branch (:488-495) with masks (:469-478), eval mode.
extern "C" int frx_decode_teacher_forced(frx_handle* h, const float* memory, const int64_t* text, int32_t B,
                                         int32_t L, float* logits, void* stream) {
  if (!h) return 1;
  const frx_config& c = h->cfg;
  if (!h->finalized) return fail(h, "teacher_forced: weights not finalized");
  if (!(h->opt_parts & 2)) return fail(h, "teacher_forced: handle was created without the decoder part");
  if (B <= 0 || B > c.max_batch) return fail(h, "teacher_forced: batch %d outside (0, %d]", B, c.max_batch);
  if (L <= 0 || L > c.max_steps || L > 500) return fail(h, "teacher_forced: length %d outside (0, %d]", L, c.max_steps);
  cudaStream_t st = (cudaStream_t)stream;
  ON_DEVICE(c.device);
  const float* A = h->arena;
  const int D = c.dec_hidden, F = c.dec_filter, V = c.num_classes, T = c.max_steps, NL = c.dec_layers;
  const int S = h->feat_h * h->feat_w, HD = D / c.dec_heads, M = B * L;
  const size_t Mm = (size_t)c.max_batch * T;
  TfWs& w = h->tf;
  if (ws_alloc(h, (void**)&w.x, Mm * D * 4) || ws_alloc(h, (void**)&w.y, Mm * D * 4) || ws_alloc(h, (void**)&w.z, Mm * D * 4) ||
      ws_alloc(h, (void**)&w.qkv, Mm * 3 * D * 4) || ws_alloc(h, (void**)&w.ff, Mm * F * 4) || ws_alloc(h, (void**)&w.mask, Mm))
    return 1;
  if (run_cross_kv(h, memory, B, st)) return 1;
  const float temp = sqrtf((float)D);
  launch_dec_embed_f32(nullptr, (const long long*)text, 0, A + h->emb, A + h->pe1d, 0, nullptr, L, temp, w.x, M, D, st);
  CKL();
  launch_pad_mask((const long long*)text, w.mask, B, L, c.pad_id, st); CKL();
  auto lin = [&](const float* in, int K, size_t wo, size_t bo, int N, float* out, int act, const float* res) {
    GemmP g = dense_gemm(in, M, K, A + wo, N, out, N);
    g.shift = A + bo; g.act = act;
    if (res) { g.res = res; g.ldr = N; }
    return g;
  };
  float* x = w.x;
  if (c.precision == FRX_PREC_BF16 && h->dec_cluster_ok && h->gen_wb) {
    // bf16 mode: every linear layer (M = B*L rows) on the tcgen05 GEMM -- bf16 operands, fp32 accumulation, fp32
    // residual stream / LayerNorm / softmax; the attention kernels are the fp32 ones (K/V history = the fp32 qkv rows).
    if (ws_alloc(h, &w.xb, Mm * D * 2) || ws_alloc(h, &w.ffb, Mm * F * 2)) return 1;
    auto tlin = [&](const void* in, int K, size_t wo, size_t bo, int N, void* out, int out_f32, int act, const float* res) {
      TcGemmP g = tc_dense(in, M, K, A, wo, N, out, out_f32);
      g.shift = A + bo; g.act = act;
      if (res) { g.res = res; g.res_f32 = 1; g.ldr = N; }
      return g;
    };
    auto to_bf16 = [&](const float* src) { launch_f32_to_h16(src, (eh_t*)w.xb, (long long)M * D, st); };
    for (int l = 0; l < NL; ++l) {
      const DecLayerW& W = h->dec[l];
      to_bf16(x); CKL();
      { TcGemmP g = tlin(w.xb, D, W.wb_sqkv, W.b_sqkv, 3 * D, w.qkv, 1, ACT_NONE, nullptr); TCL(g); }
      {
        AttnP a{};
        a.q = w.qkv; a.ldq = 3 * D; a.kcache = w.qkv + D; a.vcache = w.qkv + 2 * D; a.rows_per_img = L; a.D = 3 * D;
        a.causal_L = L; a.key_mask = w.mask; a.q_per_img = L; a.temperature = temp; a.out = w.y; a.ldo = D; a.M = M;
        a.heads = c.dec_heads;
        launch_dec_attn_f32(a, HD, st); CKL();
      }
      to_bf16(w.y); CKL();
      { TcGemmP g = tlin(w.xb, D, W.wb_o, W.b_o, D, w.z, 1, ACT_NONE, x); TCL(g); }
      launch_layernorm_f32(w.z, nullptr, A + W.ln1_g, A + W.ln1_b, w.y, M, D, 0, st); CKL();          // u -> y
      to_bf16(w.y); CKL();
      { TcGemmP g = tlin(w.xb, D, W.wb_q2, W.b_q2, D, w.z, 1, ACT_NONE, nullptr); TCL(g); }            // q2 -> z
      {
        AttnP a{};
        a.q = w.z; a.ldq = D; a.kcache = h->cross + (size_t)l * 2 * D; a.vcache = h->cross + (size_t)l * 2 * D + D;
        a.rows_per_img = S; a.D = NL * 2 * D; a.n_hist = S; a.q_per_img = L; a.temperature = temp; a.out = x; a.ldo = D;
        a.M = M; a.heads = c.dec_heads;
        launch_dec_attn_f32(a, HD, st); CKL();                                                          // c -> x (x is dead)
      }
      to_bf16(x); CKL();
      { TcGemmP g = tlin(w.xb, D, W.wb_o2, W.b_o2, D, w.z, 1, ACT_NONE, w.y); TCL(g); }
      launch_layernorm_f32(w.z, nullptr, A + W.ln2_g, A + W.ln2_b, w.y, M, D, 0, st); CKL();          // w -> y
      to_bf16(w.y); CKL();
      { TcGemmP g = tlin(w.xb, D, W.wb_f0, W.b_f0, F, w.ffb, 0, ACT_RELU, nullptr); TCL(g); }
      { TcGemmP g = tlin(w.ffb, F, W.wb_f1, W.b_f1, D, w.z, 1, ACT_RELU, w.y); TCL(g); }
      launch_layernorm_f32(w.z, nullptr, A + W.ln3_g, A + W.ln3_b, x, M, D, 0, st); CKL();            // layer output -> x
    }
    to_bf16(x); CKL();
    TcGemmP g = tc_dense(w.xb, M, D, A, h->gen_wb, V, logits, 1);
    g.shift = A + h->gen_b;
    TCL(g);
    return 0;
  }
  for (int l = 0; l < NL; ++l) {
    const DecLayerW& W = h->dec[l];
    { GemmP g = lin(x, D, W.w_sqkv, W.b_sqkv, 3 * D, w.qkv, ACT_NONE, nullptr); launch_igemm_f32(g, st); CKL(); }
    {  // masked self attention: key j <= i and not (PAD at j > 0)   (:492, :168)
      AttnP a{};
      a.q = w.qkv; a.ldq = 3 * D; a.kcache = w.qkv + D; a.vcache = w.qkv + 2 * D; a.rows_per_img = L; a.D = 3 * D;
      a.causal_L = L; a.key_mask = w.mask; a.q_per_img = L; a.temperature = temp; a.out = w.y; a.ldo = D; a.M = M;
      a.heads = c.dec_heads;
      launch_dec_attn_f32(a, HD, st); CKL();
    }
    { GemmP g = lin(w.y, D, W.w_o, W.b_o, D, w.z, ACT_NONE, x); launch_igemm_f32(g, st); CKL(); }
    launch_layernorm_f32(w.z, nullptr, A + W.ln1_g, A + W.ln1_b, w.y, M, D, 0, st); CKL();          // u -> y
    { GemmP g = lin(w.y, D, W.w_q2, W.b_q2, D, w.z, ACT_NONE, nullptr); launch_igemm_f32(g, st); CKL(); }  // q2 -> z
    {
      AttnP a{};
      a.q = w.z; a.ldq = D; a.kcache = h->cross + (size_t)l * 2 * D; a.vcache = h->cross + (size_t)l * 2 * D + D;
      a.rows_per_img = S; a.D = NL * 2 * D; a.n_hist = S; a.q_per_img = L; a.temperature = temp; a.out = x; a.ldo = D;
      a.M = M; a.heads = c.dec_heads;
      launch_dec_attn_f32(a, HD, st); CKL();                                                          // c -> x (x is dead)
    }
    { GemmP g = lin(x, D, W.w_o2, W.b_o2, D, w.z, ACT_NONE, w.y); launch_igemm_f32(g, st); CKL(); }
    launch_layernorm_f32(w.z, nullptr, A + W.ln2_g, A + W.ln2_b, w.y, M, D, 0, st); CKL();          // w -> y
    { GemmP g = lin(w.y, D, W.w_f0, W.b_f0, F, w.ff, ACT_RELU, nullptr); launch_igemm_f32(g, st); CKL(); }
    { GemmP g = lin(w.ff, F, W.w_f1, W.b_f1, D, w.z, ACT_RELU, w.y); launch_igemm_f32(g, st); CKL(); }
    launch_layernorm_f32(w.z, nullptr, A + W.ln3_g, A + W.ln3_b, x, M, D, 0, st); CKL();            // layer output -> x
  }
  GemmP g = dense_gemm(x, M, D, A + h->gen_w, V, logits, V);
  g.shift = A + h->gen_b;
  launch_igemm_f32(g, st); CKL();
  return 0;
}

// Test / micro-benchmark hook for the tcgen05 implicit-GEMM kernel (see include/frx.h).
extern "C" int frx_tc_gemm(frx_handle* h, const void* A, const void* W, void* C, int32_t M, int32_t N, int32_t K,
                           const int32_t* conv7, const float* scale, const float* shift, int32_t act,
                           int32_t out_f32, void* stream) {
  if (!h) return 1;
  cudaStream_t st = (cudaStream_t)stream;
  ON_DEVICE(h->cfg.device);
  TcGemmP g{};
  g.A = (const eh_t*)A; g.W = (const eh_t*)W; g.C = C;
  g.M = M; g.N = N; g.K = K; g.lda = K; g.ldw = K; g.ldc = N; g.out_f32 = out_f32;
  g.scale = scale; g.shift = shift; g.act = act;
  if (conv7) {  // {B, H, W, Cin, ksize, stride, same_pad(1) or zero pad(0)}
    int B = conv7[0], H = conv7[1], Wd = conv7[2], Cin = conv7[3], k = conv7[4], s = conv7[5];
    int OH, OW, pt = 0, pl = 0;
    if (conv7[6]) { same_pad(H, k, s, &OH, &pt); same_pad(Wd, k, s, &OW, &pl); }
    else { OH = (H - k) / s + 1; OW = (Wd - k) / s + 1; }
    if (M != B * OH * OW || K != k * k * Cin) return fail(h, "frx_tc_gemm: conv shape mismatch (M %d vs %d, K %d vs %d)", M, B * OH * OW, K, k * k * Cin);
    g.conv = 1; g.H = H; g.Wd = Wd; g.Cin = Cin; g.OH = OH; g.OW = OW; g.KW = k; g.stride = s; g.pad_t = pt; g.pad_l = pl;
    if (h->opt_tc_ws && h->opt_tc_im2col && Cin <= 64) {
      size_t bytes = (size_t)N * k * k * 64 * 2;
      if (h->hook_wpad_bytes < bytes) {
        void* q;
        if (dev_alloc(h, &q, bytes)) return 1;
        h->hook_wpad = q; h->hook_wpad_bytes = bytes;
      }
      launch_pad_conv_weights((const eh_t*)W, (eh_t*)h->hook_wpad, (long long)N * k * k, Cin, st); CKL();
      g.Wpad = (const eh_t*)h->hook_wpad;
    }
  }
  TCL(g);
  return 0;
}
