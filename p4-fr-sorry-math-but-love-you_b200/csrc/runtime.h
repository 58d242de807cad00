// runtime.h -- the handle behind include/frx.h (host-side state only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <map>
#include <string>
#include <tuple>
#include <vector>

#include "../../include/frx.h"

struct HostTensor {
  std::vector<int64_t> shape;
  std::vector<float> f;
};

// Offsets (in floats) into the weight arena.
struct BlockW {
  int kind;  // 0 ConvBnAct, 1 EdgeResidual (fused-MBConv), 2 InvertedResidual (MBConv + SE)
  int cin, cout, k, stride, mid, se_r;
  bool residual;
  std::string name;
  size_t w_a, sc_a, sh_a;      // first conv (3x3 for kinds 0/1, 1x1 expand for kind 2) + folded BN
  size_t w_dw, sc_dw, sh_dw;   // depthwise 3x3 + folded BN (kind 2)
  size_t se_w1, se_b1, se_w2, se_b2, se_w2t = 0;
  size_t w_b, sc_b, sh_b;      // 1x1 projection + folded BN (kinds 1/2)
  size_t wb_a = 0, wb_b = 0;   // bf16 copies of w_a / w_b ([N][K], K contiguous) for the tcgen05 path
  size_t wb_a_pad = 0;         // 3x3 convs: bf16 [N][9][64] (channels zero-padded) for the TMA-im2col path
  size_t w_frag24 = 0;         // 24 -> 24 3x3 convs: mma.m16n8k16 B fragments [14][3][32] x {b0, b1} (conv3x3_c24_mma_kernel)
};
struct LiteConvW { int cin, cout; size_t w, sc, sh; size_t wb = 0; };  // wb: bf16 copy of w (layers 1-3, bf16 mode)
struct EncLayerW {
  size_t ln_g, ln_b, w_qkv, b_qkv, w_o, b_o;
  size_t w_c0, sc_c0, sh_c0, w_dw, sc_dw, sh_dw, w_c1, sc_c1, sh_c1;
  size_t wb_qkv = 0, wb_o = 0, wb_c0 = 0, wb_c1 = 0;   // bf16 copies
};
struct DecLayerW {
  size_t wt_o, b_o, wt_q2, b_q2, wt_o2, b_o2, wt_f0, b_f0, wt_f1, b_f1;   // [K][N] for the step kernels
  size_t w_o, w_q2, w_o2, w_f0, w_f1, w_sqkv, b_sqkv;                     // [N][K] for the teacher-forced path
  size_t wb_o = 0, wb_q2 = 0, wb_o2 = 0, wb_f0 = 0, wb_f1 = 0, wb_sqkv = 0;  // bf16 copies of the above (bf16 mode)
  size_t ln1_g, ln1_b, ln2_g, ln2_b, ln3_g, ln3_b;
};
struct FusedW { size_t wt, b; int N; };
struct SwinBlockW {
  int dim, res, heads, ws, shift;
  size_t n1_g, n1_b, bias_table, qkv_w, qkv_b, proj_w, proj_b, n2_g, n2_b, fc1_w, fc1_b, fc2_w, fc2_b;
  size_t qkv_wb = 0, proj_wb = 0, fc1_wb = 0, fc2_wb = 0;  // bf16 copies (bf16 mode)
};
struct SwinMergeW { int dim, res; size_t red_w, n_g, n_b; size_t red_wb = 0; };
// fragment-packed bf16 weights of the persistent decode kernel (offsets in floats = u32 words)
struct DecPackW { size_t w_o, w_q2, w_o2, w_f0, w_f1, w_next; };
struct Tap { float* data = nullptr; size_t capacity = 0; int shape[4] = {0, 0, 0, 0}; };
typedef std::tuple<int, int, int> GraphKey;  // batch, steps, mode (0 greedy, 1 forced, 2 DecodingManager)
struct GraphEntry { cudaGraphExec_t exec; int64_t nodes; int64_t last_use = 0; };
constexpr size_t FRX_MAX_GRAPHS = 4;   // least-recently-used eviction beyond this many captured decode loops

struct BeamWs {
  double *hscore = nullptr, *nlogp = nullptr;
  int *hnode = nullptr, *nprev = nullptr, *ntok = nullptr, *nlen = nullptr, *nkv = nullptr, *chain = nullptr, *small = nullptr;
  float* logits = nullptr;
  int* host_flag = nullptr;
};
struct TfWs {
  float *x = nullptr, *y = nullptr, *z = nullptr, *qkv = nullptr, *ff = nullptr;
  unsigned char* mask = nullptr;
  void *xb = nullptr, *ffb = nullptr;  // bf16 A operands of the tcgen05 GEMMs (bf16 mode)
};

struct frx_handle {
  frx_config cfg{};
  std::string err;
  int num_sms = 0;
  std::map<std::string, HostTensor> raw;
  bool finalized = false, ws_ready = false;
  bool opt_taps = false, opt_graphs = true, opt_timing = false, opt_step16 = true, opt_pipe_enc = true;
  int* step_hist = nullptr;   // [max_batch] history length of the step_forward state (cluster kernel in step mode)
  bool opt_prof = false;
  bool opt_tc_im2col = true;   // 3x3 conv A tiles by TMA im2col (false: cp.async gather)
  void* hook_wpad = nullptr; size_t hook_wpad_bytes = 0;
  bool opt_tc_ws = true;       // persistent warp-specialised tcgen05 GEMM (false: one tile per CTA)
  int opt_dec_hpc = 0;         // 256-wide bf16 decode kernel: heads per CTA (2: clusters of 4 x 16 warps, 1: clusters of 8 x 8 warps, 0: by batch)
  bool opt_conv24 = true;      // stage-0 24 -> 24 convs on the halo-tile mma.sync kernel (false: tcgen05 im2col GEMM)
  bool opt_enc_fp32 = false;   // bf16 handle, but run the encoder on the fp32 SIMT path (debug)
  long long* prof = nullptr;
  int opt_parts = 3;  // bit0: encoder weights/workspaces, bit1: decoder
  int feat_h = 0, feat_w = 0;
  std::vector<void*> allocs;
  int64_t device_bytes = 0, launches = 0;

  float* arena = nullptr;
  size_t arena_bytes = 0;
  // trunk
  size_t stem_w = 0, stem_sc = 0, stem_sh = 0, last_w = 0, last_sc = 0, last_sh = 0;
  std::vector<BlockW> blocks;
  LiteConvW lite[4]{};
  // encoder
  size_t pe_w0 = 0, pe_b0 = 0, pe_w1 = 0, pe_b1 = 0, pe_h = 0, pe_w = 0;
  std::vector<EncLayerW> enc;
  // SwinTRN encoder
  size_t sw_pe_w = 0, sw_pe_b = 0, sw_pe_g = 0, sw_pe_beta = 0, sw_ape = 0, sw_norm_g = 0, sw_norm_b = 0;
  std::vector<SwinBlockW> sw_blocks;
  std::vector<SwinMergeW> sw_merges;   // merge i follows the last block of stage i
  float *sw_x[2] = {nullptr, nullptr}, *sw_a = nullptr, *sw_qkv = nullptr, *sw_hid = nullptr;
  // decoder
  size_t emb = 0, pe1d = 0, gen_w = 0, gen_b = 0, w_cross = 0, b_cross = 0;
  size_t gen_wb = 0;  // bf16 copy of the generator weight (teacher-forced path, bf16 mode)
  size_t last_wb = 0, cross_wb = 0;   // bf16 copies of conv_last / cross K|V weights
  std::vector<DecLayerW> dec;
  std::vector<FusedW> fused;
  std::vector<DecPackW> dpack;
  size_t dpack_first = 0;
  std::vector<DecPackW> dpack2;   // 256-wide decoder packed for two heads per CTA (clusters of 4)
  size_t dpack2_first = 0;

  // workspaces
  float *act[2] = {nullptr, nullptr}, *mid[2] = {nullptr, nullptr}, *gate = nullptr;
  float *kself = nullptr, *vself = nullptr, *cross = nullptr;
  float *dx = nullptr, *dqkv = nullptr, *datt = nullptr, *dpre1 = nullptr, *dpre2 = nullptr, *du = nullptr,
        *dw = nullptr, *dq2 = nullptr, *dff = nullptr;
  float *logits_int = nullptr, *memory_int = nullptr, *images_int = nullptr;
  long long *tokens_int = nullptr, *forced_int = nullptr;
  int* cur_tok = nullptr;
  int* eos_work = nullptr;       // work counter of the stop-at-<EOS> decode kernel
  void* mem_bf = nullptr;  // bf16 copy of the encoder memory (A operand of the cross K/V GEMM)
  void *kself_bf = nullptr, *vself_bf = nullptr, *kcross_bf = nullptr, *vcross_bf = nullptr;  // bf16 caches

  std::map<GraphKey, GraphEntry> graphs;
  int64_t graph_clock = 0;
  std::map<std::string, Tap> taps;
  cudaEvent_t ev[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};
  // pipelined host entry (frx_forward_greedy_host_submit / _wait): two staging slots, one stream per copy direction
  struct PipeSlot {
    float *img = nullptr, *mem = nullptr;   // staged images, this batch's encoder output
    long long* tok = nullptr;
    cudaEvent_t h2d = nullptr, enc = nullptr, done = nullptr, d2h = nullptr;
    bool busy = false;
  };
  PipeSlot pipe[2];
  cudaStream_t pipe_h2d = nullptr, pipe_d2h = nullptr, pipe_enc = nullptr;
  float last_ms[4] = {0, 0, 0, 0};
  BeamWs beam;
  TfWs tf;
  int step_idx = 0, step_batch = 0;
  // DecodingManager rule tables (frx_set_decoding_rules) and per-row state of the constrained greedy decode
  int *sift_flags = nullptr, *sift_limit = nullptr;
  int4* sift_state = nullptr;
  int sift_ids[6] = {0, 0, 0, 0, 0, 0};  // <SOS>, <EOS>, "", "{", "}", "_"
  bool have_rules = false;
  bool timed_kernel = false;
  bool opt_train_splitk = true;   // training step: deterministic split-K for the GEMM launches of few tiles (train.cu)
  bool dec_cluster_ok = false;   // bf16 mode: the persistent cluster decode kernel fits this decoder's dimensions
  void* train = nullptr;   // TrainState (train.cu): parameters, gradients, optimiser state of the training step
  void *sw_ab = nullptr, *sw_hidb = nullptr;  // SwinTRN bf16 mode: bf16 A operands (LayerNorm / attention output, MLP hidden)
};
