// train_kernels.h -- launchers of the training-step kernels (kernels_train.cu).
#pragma once
#include <cuda_runtime.h>

#include "common.cuh"

namespace frx {

// dW[n][k] += sum_m dZ[m][n] * A(m, k); A dense [M, lda] or an NHWC activation gathered with the forward geometry
struct WgradP {
  const float* dZ;   // [M, ldz]
  const float* A;
  float* dW;         // [N][K]
  long long M;
  int N, K, ldz, lda;
  int conv, H, Wd, Cin, OH, OW, KW, stride, pad_t, pad_l;
  long long m_chunk;  // set by the launcher
};

struct AttnBwdP {
  const float *q, *k, *v, *dout;
  float *dq, *dk, *dv;
  int ldq, ldk, ldv, ldo, lddq, lddk, lddv;
  int Lq, Lk, heads, HD;
  int causal;
  const unsigned char* key_mask;   // [B][Lk] or nullptr
  float temperature;
  int accumulate_kv;               // dk / dv += instead of =
  DropP drop;                      // attention dropout of the forward pass (drop.step == nullptr: none)
};

void launch_fill(float* p, float v, long long n, cudaStream_t st);
void launch_axpy(float* y, const float* x, float a, long long n, int accumulate, cudaStream_t st);
void launch_act_fwd(const float* in, float* out, int act, long long n, cudaStream_t st);
void launch_act_bwd(const float* dout, const float* pre, float* din, int act, long long n, cudaStream_t st);
void launch_repack_dgrad(const float* w, float* out, int R, int T, int C, cudaStream_t st);
void launch_zero_stuff(const float* dz, float* z, int B, int OH, int OW, int C, int s, int ZH, int ZW, cudaStream_t st);
void launch_scramble(const float* in, float* out, int B, int S, int C, int inverse, cudaStream_t st);
void launch_bn_stats(const float* z, double* acc, const float* gamma, const float* beta, float* running_mean, float* running_var, float* stat,
                     int M, int C, float eps, float momentum, cudaStream_t st);
void launch_bn_apply(const float* z, const float* stat, const float* res, float* y, long long M, int C, int act, cudaStream_t st);
void launch_bn_bwd(const float* dy, const float* z, const float* stat, double* acc, float* dz, float* dgamma, float* dbeta, int M, int C,
                   int act, cudaStream_t st);
void launch_wgrad(WgradP p, int num_sms, cudaStream_t st);
void launch_colsum(const float* dz, float* db, long long M, int C, int ld, cudaStream_t st);
void launch_dw_bwd(const float* dz, const float* x, const float* w, float* dx, float* dw, float* db, int B, int H, int W, int C, int OH, int OW,
                   int stride, int pad_t, int pad_l, cudaStream_t st);
void launch_spatial_dot(const float* a, const float* b2, float* out, int B, int S, int C, float scale, cudaStream_t st);
void launch_spatial_scale(const float* x, const float* g, const float* add, float* out, int B, int S, int C, cudaStream_t st);
void launch_spatial_add(float* x, const float* add, int B, int S, int C, float scale, cudaStream_t st);
void launch_pe2d_apply(const float* x, const float* g, const float* peh, const float* pew, float* out, int B, int h, int w, int C,
                       const DropP& drop, cudaStream_t st);
void launch_dropout(const float* x, const float* add, float* y, long long n, const DropP& d, int S, int C, cudaStream_t st);
void launch_counter_add(uint32_t* ctr, uint32_t v, cudaStream_t st);
void launch_philox_probe(uint4* io, cudaStream_t st);
void launch_pe2d_bwd_gate(const float* dout, const float* peh, const float* pew, float* dg, int B, int h, int w, int C, cudaStream_t st);
void launch_ln_fwd(const float* x, const float* gamma, const float* beta, float* y, float* stat, int M, int C, cudaStream_t st);
void launch_ln_bwd(const float* dy, const float* x, const float* stat, const float* gamma, float* dx, float* dgamma, float* dbeta, int M, int C,
                   cudaStream_t st);
int launch_attn_bwd(const AttnBwdP& p, int B, cudaStream_t st);
void launch_embed_bwd(const long long* tok, const float* dx, float* dE, int M, int D, float scale, cudaStream_t st);
void launch_cross_entropy(const float* logits, const long long* expected, float* dlogits, float* out2, int B, int L, int V, int pad, cudaStream_t st);
void launch_stem_wgrad(const float* dz, const float* img, float* dw, int B, int Cin, int H, int W, int OH, int OW, int Cout, cudaStream_t st);
int launch_image_conv_wgrad(const float* dz, const float* img, float* dw, int B, int Cin, int H, int W, int OH, int OW, int Cout, int stride,
                            int pad, cudaStream_t st);
void launch_maxpool2_fwd(const float* x, float* y, int B, int H, int W, int C, cudaStream_t st);
void launch_maxpool2_bwd(const float* x, const float* dy, float* dx, int B, int H, int W, int C, cudaStream_t st);
void launch_sumsq(const float* g, long long n, double* out, cudaStream_t st);
void launch_adamw(float* p, const float* g, float* m, float* v, const double* sumsq, float* norm_out, long long n, float lr, float wd, int step,
                  float max_norm, float grad_scale, cudaStream_t st);

}  // namespace frx
