// kernels_train.cu -- kernels of the teacher-forced TRAINING step (train_modules/train_single_opt.py:72-112):
// train-mode BatchNorm (batch statistics) forward / backward, weight-gradient contractions, depthwise / squeeze-excite /
// LayerNorm / attention backward, cross-entropy with ignore_index, gradient-norm clipping and AdamW.
//
// All arithmetic is fp32 (the reference trains in fp32: GradScaler is constructed at train_single_opt.py:413 and never
// used, no autocast).  Activations are NHWC = row-major [rows, channels] like the inference path; forward contractions
// and the data gradients of convolutions / linear layers re-use the fp32 implicit-GEMM kernel of kernels_f32.cu (the
// data gradient of a convolution is a convolution of the zero-stuffed output gradient with the flipped, transposed
// filter).  Reductions over the batch (BatchNorm statistics, weight gradients, bias gradients) accumulate per-CTA
// partial sums with atomics: the summation order is not fixed, results agree with the reference to fp32 round-off.
#include "common.cuh"
#include "kernels.h"
#include "train_kernels.h"

namespace frx {

namespace {

__device__ __forceinline__ float act_grad(float u, int act) {   // d act(u) / du
  if (act == ACT_RELU) return u > 0.f ? 1.f : 0.f;
  if (act == ACT_SILU) {
    const float s = 1.f / (1.f + expf(-u));
    return s * (1.f + u * (1.f - s));
  }
  if (act == ACT_SIGMOID) {
    const float s = 1.f / (1.f + expf(-u));
    return s * (1.f - s);
  }
  return 1.f;
}

__device__ __forceinline__ double warp_sum_d(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

}  // namespace

// =====================================================================================================================
// elementwise helpers
// =====================================================================================================================
__global__ void __launch_bounds__(256) fill_kernel(float* p, float v, long long n) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) p[i] = v;
}
void launch_fill(float* p, float v, long long n, cudaStream_t st) {
  if (n > 0) fill_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(p, v, n);
}

// y = a * x (+ y)
__global__ void __launch_bounds__(256) axpy_kernel(float* __restrict__ y, const float* __restrict__ x, float a, long long n, int accumulate) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) y[i] = accumulate ? fmaf(a, x[i], y[i]) : a * x[i];
}
void launch_axpy(float* y, const float* x, float a, long long n, int accumulate, cudaStream_t st) {
  if (n > 0) axpy_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(y, x, a, n, accumulate);
}

// dropout: y = x * M * scale (+ add).  Element i of the row-major buffer has the logical index i, or with S > 0 the buffer
// is NHWC [B, S, C] and the logical layout NCHW [B, C, S].  In place (y == x) is allowed.
__global__ void __launch_bounds__(256) dropout_kernel(const float* x, const float* __restrict__ add, float* y, long long n, const DropP d, int S,
                                                      int C) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  long long e = i;
  if (S > 0) {
    const long long b = i / ((long long)S * C);
    const int c = (int)(i % C), q = (int)((i / C) % S);
    e = (b * C + c) * S + q;
  }
  const float v = __fmul_rn(x[i], drop_factor(d, e));
  y[i] = add ? __fadd_rn(v, add[i]) : v;
}
void launch_dropout(const float* x, const float* add, float* y, long long n, const DropP& d, int S, int C, cudaStream_t st) {
  if (n > 0) dropout_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(x, add, y, n, d, S, C);
}
// the dropout step counter: *ctr += v (one thread)
__global__ void counter_add_kernel(uint32_t* ctr, uint32_t v) { *ctr += v; }
void launch_counter_add(uint32_t* ctr, uint32_t v, cudaStream_t st) { counter_add_kernel<<<1, 1, 0, st>>>(ctr, v); }
// philox4x32_10 of one counter / key (the test hook frx_philox4x32)
__global__ void philox_probe_kernel(uint4* io) { io[0] = philox4x32_10(io[0], make_uint2(io[1].x, io[1].y)); }
void launch_philox_probe(uint4* io, cudaStream_t st) { philox_probe_kernel<<<1, 1, 0, st>>>(io); }

// out = act(in); dgrad variant: out = dout * act'(pre)
__global__ void __launch_bounds__(256) act_fwd_kernel(const float* __restrict__ in, float* __restrict__ out, int act, long long n) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = act_apply(in[i], act);
}
void launch_act_fwd(const float* in, float* out, int act, long long n, cudaStream_t st) {
  act_fwd_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(in, out, act, n);
}
__global__ void __launch_bounds__(256) act_bwd_kernel(const float* __restrict__ dout, const float* __restrict__ pre, float* __restrict__ din, int act, long long n) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) din[i] = dout[i] * act_grad(pre[i], act);
}
void launch_act_bwd(const float* dout, const float* pre, float* din, int act, long long n, cudaStream_t st) {
  act_bwd_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(dout, pre, din, act, n);
}

// [R][T][C] -> [C][T'][R] with T' = T-1-t (filter flip); T = 1: plain transpose.  Used for the data gradients:
// W [Cout][taps][Cin] -> W' [Cin][flipped taps][Cout];  linear W [N][K] -> [K][N].
__global__ void __launch_bounds__(256) repack_dgrad_kernel(const float* __restrict__ w, float* __restrict__ out, int R, int T, int C) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (long long)R * T * C) return;
  const int r = (int)(i % R);
  const int t = (int)((i / R) % T);
  const int c = (int)(i / ((long long)R * T));
  out[i] = w[((long long)r * T + (T - 1 - t)) * C + c];
}
void launch_repack_dgrad(const float* w, float* out, int R, int T, int C, cudaStream_t st) {
  long long n = (long long)R * T * C;
  repack_dgrad_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(w, out, R, T, C);
}

// zero-stuffing of an output gradient for the data gradient of a strided convolution: Z[n][oh*s][ow*s][c] = dz[n][oh][ow][c]
__global__ void __launch_bounds__(256) zero_stuff_kernel(const float* __restrict__ dz, float* __restrict__ z, int B, int OH, int OW, int C, int s,
                                                         int ZH, int ZW) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (long long)B * OH * OW * C) return;
  const int c = (int)(i % C);
  long long pix = i / C;
  const int ow = (int)(pix % OW), oh = (int)((pix / OW) % OH), n = (int)(pix / ((long long)OW * OH));
  z[(((long long)n * ZH + oh * s) * ZW + ow * s) * C + c] = dz[i];
}
void launch_zero_stuff(const float* dz, float* z, int B, int OH, int OW, int C, int s, int ZH, int ZW, cudaStream_t st) {
  cudaMemsetAsync(z, 0, (size_t)B * ZH * ZW * C * 4, st);
  long long n = (long long)B * OH * OW * C;
  zero_stuff_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(dz, z, B, OH, OW, C, s, ZH, ZW);
}

// the reference's raw reshape (EfficientSATRN.py:269, SURVEY F4) as a per-image permutation of S*C elements:
// forward: out[pp*C + cc] = in[f], f = cc*S + pp;  inverse (gradients): out[f] = in[pp*C + cc]
__global__ void __launch_bounds__(256) scramble_kernel(const float* __restrict__ in, float* __restrict__ out, int S, int C, long long n, int inverse) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const long long img = i / ((long long)S * C);
  const int g = (int)(i % ((long long)S * C));
  const int pp = g / C, cc = g % C;
  const long long f = img * S * C + (long long)cc * S + pp;
  if (inverse) out[f] = in[i];
  else out[i] = in[f];
}
void launch_scramble(const float* in, float* out, int B, int S, int C, int inverse, cudaStream_t st) {
  long long n = (long long)B * S * C;
  scramble_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(in, out, S, C, n, inverse);
}

// =====================================================================================================================
// BatchNorm, train mode (nn.BatchNorm2d.forward with self.training): batch statistics over the M = B*H*W rows
// =====================================================================================================================
// per-channel sum / sum of squares around a per-channel pivot (row 0): 32 channels x 8 row lanes per CTA
__global__ void __launch_bounds__(256) bn_stats_kernel(const float* __restrict__ z, double* __restrict__ acc /*[C][2]*/, int M, int C, int rows_per_cta) {
  const int cl = threadIdx.x & 31, rl = threadIdx.x >> 5;
  const int c = blockIdx.x * 32 + cl;
  const int r0 = blockIdx.y * rows_per_cta;
  const int r1 = min(M, r0 + rows_per_cta);
  float s = 0.f, q = 0.f;
  const float pivot = c < C ? __ldg(z + c) : 0.f;
  if (c < C)
    for (int r = r0 + rl; r < r1; r += 8) {
      const float d = __ldg(z + (long long)r * C + c) - pivot;
      s += d;
      q = fmaf(d, d, q);
    }
  __shared__ float ss[8][33], qq[8][33];
  ss[rl][cl] = s; qq[rl][cl] = q;
  __syncthreads();
  if (rl == 0 && c < C) {
    double S = 0, Q = 0;
#pragma unroll
    for (int i = 0; i < 8; ++i) { S += ss[i][cl]; Q += qq[i][cl]; }
    atomicAdd(acc + 2 * c, S);
    atomicAdd(acc + 2 * c + 1, Q);
  }
}
// statistics -> (mean, invstd), folded (alpha, beta), running statistics update (momentum, unbiased variance)
__global__ void __launch_bounds__(256) bn_finalize_kernel(const float* __restrict__ z, const double* __restrict__ acc, const float* __restrict__ gamma,
                                                          const float* __restrict__ beta, float* __restrict__ running_mean,
                                                          float* __restrict__ running_var, float* __restrict__ stat /*[4][C]: mean, invstd, alpha, beta*/,
                                                          int M, int C, float eps, float momentum) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  const double pivot = z[c];
  const double md = acc[2 * c] / M;
  const double mean = pivot + md;
  double var = acc[2 * c + 1] / M - md * md;
  if (var < 0) var = 0;
  const float invstd = (float)(1.0 / sqrt(var + (double)eps));
  const float a = gamma[c] * invstd;
  stat[c] = (float)mean;
  stat[C + c] = invstd;
  stat[2 * C + c] = a;
  stat[3 * C + c] = beta[c] - (float)mean * a;
  if (running_mean) {
    const double unbiased = M > 1 ? var * M / (M - 1) : var;
    running_mean[c] = (1.f - momentum) * running_mean[c] + momentum * (float)mean;
    running_var[c] = (1.f - momentum) * running_var[c] + momentum * (float)unbiased;
  }
}
void launch_bn_stats(const float* z, double* acc, const float* gamma, const float* beta, float* running_mean, float* running_var, float* stat,
                     int M, int C, float eps, float momentum, cudaStream_t st) {
  cudaMemsetAsync(acc, 0, (size_t)C * 2 * sizeof(double), st);
  int chunks = (M + 511) / 512;
  if (chunks > 1024) chunks = 1024;
  const int rows = (M + chunks - 1) / chunks;
  bn_stats_kernel<<<dim3((C + 31) / 32, (M + rows - 1) / rows), 256, 0, st>>>(z, acc, M, C, rows);
  bn_finalize_kernel<<<(C + 255) / 256, 256, 0, st>>>(z, acc, gamma, beta, running_mean, running_var, stat, M, C, eps, momentum);
}

// y = act(z * alpha + beta) (+ res)
__global__ void __launch_bounds__(256) bn_apply_kernel(const float* __restrict__ z, const float* __restrict__ stat, const float* __restrict__ res,
                                                       float* __restrict__ y, long long n4, int C, int act) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n4) return;
  const int c = (int)((i * 4) % C);
  const float4 v = __ldg(reinterpret_cast<const float4*>(z) + i);
  const float4 a = __ldg(reinterpret_cast<const float4*>(stat + 2 * C + c)), b = __ldg(reinterpret_cast<const float4*>(stat + 3 * C + c));
  float4 o = make_float4(act_apply(fmaf(v.x, a.x, b.x), act), act_apply(fmaf(v.y, a.y, b.y), act), act_apply(fmaf(v.z, a.z, b.z), act),
                         act_apply(fmaf(v.w, a.w, b.w), act));
  if (res) {
    const float4 r = __ldg(reinterpret_cast<const float4*>(res) + i);
    o.x += r.x; o.y += r.y; o.z += r.z; o.w += r.w;
  }
  reinterpret_cast<float4*>(y)[i] = o;
}
void launch_bn_apply(const float* z, const float* stat, const float* res, float* y, long long M, int C, int act, cudaStream_t st) {
  const long long n4 = M * C / 4;
  bn_apply_kernel<<<(unsigned)((n4 + 255) / 256), 256, 0, st>>>(z, stat, res, y, n4, C, act);
}

// backward, pass 1: du = dy * act'(u), u = z*alpha+beta; per-channel sums of du and du * zhat
__global__ void __launch_bounds__(256) bn_bwd_reduce_kernel(const float* __restrict__ dy, const float* __restrict__ z, const float* __restrict__ stat,
                                                            double* __restrict__ acc, int M, int C, int act, int rows_per_cta) {
  const int cl = threadIdx.x & 31, rl = threadIdx.x >> 5;
  const int c = blockIdx.x * 32 + cl;
  const int r0 = blockIdx.y * rows_per_cta, r1 = min(M, r0 + rows_per_cta);
  float s = 0.f, q = 0.f;
  if (c < C) {
    const float mean = stat[c], invstd = stat[C + c], a = stat[2 * C + c], b = stat[3 * C + c];
    for (int r = r0 + rl; r < r1; r += 8) {
      const float zz = __ldg(z + (long long)r * C + c);
      const float du = __ldg(dy + (long long)r * C + c) * act_grad(fmaf(zz, a, b), act);
      s += du;
      q = fmaf(du, (zz - mean) * invstd, q);
    }
  }
  __shared__ float ss[8][33], qq[8][33];
  ss[rl][cl] = s; qq[rl][cl] = q;
  __syncthreads();
  if (rl == 0 && c < C) {
    double S = 0, Q = 0;
#pragma unroll
    for (int i = 0; i < 8; ++i) { S += ss[i][cl]; Q += qq[i][cl]; }
    atomicAdd(acc + 2 * c, S);
    atomicAdd(acc + 2 * c + 1, Q);
  }
}
// pass 2: dz = gamma*invstd * (du - sum(du)/M - zhat * sum(du*zhat)/M); dgamma += sum(du*zhat), dbeta += sum(du)
__global__ void __launch_bounds__(256) bn_bwd_apply_kernel(const float* __restrict__ dy, const float* __restrict__ z, const float* __restrict__ stat,
                                                           const double* __restrict__ acc, float* __restrict__ dz, long long n, int M, int C, int act) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int c = (int)(i % C);
  const float mean = stat[c], invstd = stat[C + c], a = stat[2 * C + c], b = stat[3 * C + c];
  const float zz = z[i];
  const float du = dy[i] * act_grad(fmaf(zz, a, b), act);
  const float zh = (zz - mean) * invstd;
  const float sdu = (float)(acc[2 * c] / M), sdz = (float)(acc[2 * c + 1] / M);
  dz[i] = a * (du - sdu - zh * sdz);   // a = gamma * invstd
}
__global__ void __launch_bounds__(256) bn_bwd_params_kernel(const double* __restrict__ acc, float* __restrict__ dgamma, float* __restrict__ dbeta, int C) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  dgamma[c] += (float)acc[2 * c + 1];
  dbeta[c] += (float)acc[2 * c];
}
void launch_bn_bwd(const float* dy, const float* z, const float* stat, double* acc, float* dz, float* dgamma, float* dbeta, int M, int C,
                   int act, cudaStream_t st) {
  cudaMemsetAsync(acc, 0, (size_t)C * 2 * sizeof(double), st);
  // rows per CTA: 512 for the large early-stage maps; for the small late-stage ones (M = 512 rows at 16 images) one CTA
  // per 32 channels would walk all rows serially (41 us for 6 MB): split the rows until ~600 CTAs exist (the per-CTA
  // partial sums meet in fp64 atomics either way)
  int chunks = (M + 511) / 512;
  const int cgroups = (C + 31) / 32;
  if (cgroups * chunks < 600) chunks = (600 + cgroups - 1) / cgroups;
  if (chunks > (M + 31) / 32) chunks = (M + 31) / 32;
  if (chunks > 1024) chunks = 1024;
  if (chunks < 1) chunks = 1;
  const int rows = (M + chunks - 1) / chunks;
  bn_bwd_reduce_kernel<<<dim3(cgroups, (M + rows - 1) / rows), 256, 0, st>>>(dy, z, stat, acc, M, C, act, rows);
  const long long n = (long long)M * C;
  bn_bwd_apply_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(dy, z, stat, acc, dz, n, M, C, act);
  bn_bwd_params_kernel<<<(C + 255) / 256, 256, 0, st>>>(acc, dgamma, dbeta, C);
}

// =====================================================================================================================
// weight gradient: dW[n][k] += sum_m dZ[m][n] * A(m, k), A dense [M, lda] or gathered from NHWC (conv forward geometry).
// CTA tile 64 x 64 outputs over an m-range; 16-row slabs of dZ and A in shared memory; 4 x 4 outputs per thread.
// =====================================================================================================================
__global__ void __launch_bounds__(256) wgrad_kernel(const WgradP p) {
  constexpr int BM = 16;
  __shared__ __align__(16) float Zs[BM][64 + 4];
  __shared__ __align__(16) float As[BM][64 + 4];
  const int tid = threadIdx.x;
  const int n0 = blockIdx.x * 64, k0 = blockIdx.y * 64;
  const long long m_begin = (long long)blockIdx.z * p.m_chunk;
  const long long m_end = m_begin + p.m_chunk < p.M ? m_begin + p.m_chunk : p.M;
  const int lr = tid >> 4, lc = (tid & 15) * 4;   // loader: row lr of the slab, 4 consecutive columns from lc
  const int tx = tid & 15, ty = tid >> 4;         // compute: n rows ty*4.., k columns tx*4..
  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
  // conv gather: column k = (tap, ci); a 4-aligned k group never straddles a tap (Cin % 4 == 0)
  const int kk = k0 + lc;
  int tap = 0, ci = kk, kh = 0, kw = 0;
  if (p.conv) { tap = kk / p.Cin; ci = kk - tap * p.Cin; kh = tap / p.KW; kw = tap - kh * p.KW; }
  for (long long m0 = m_begin; m0 < m_end; m0 += BM) {
    const long long m = m0 + lr;
    float4 zv = make_float4(0.f, 0.f, 0.f, 0.f), av = zv;
    if (m < m_end) {
      const int n = n0 + lc;
      if (n + 3 < p.N && (p.ldz & 3) == 0) zv = __ldg(reinterpret_cast<const float4*>(p.dZ + m * p.ldz + n));
      else {
        float t[4] = {0.f, 0.f, 0.f, 0.f};
        for (int i = 0; i < 4; ++i) if (n + i < p.N) t[i] = __ldg(p.dZ + m * p.ldz + n + i);
        zv = make_float4(t[0], t[1], t[2], t[3]);
      }
      if (kk < p.K) {
        if (p.conv) {
          const int ow = (int)(m % p.OW);
          const long long t = m / p.OW;
          const int oh = (int)(t % p.OH);
          const long long img = t / p.OH;
          const int ih = oh * p.stride - p.pad_t + kh, iw = ow * p.stride - p.pad_l + kw;
          if (ih >= 0 && ih < p.H && iw >= 0 && iw < p.Wd)
            av = __ldg(reinterpret_cast<const float4*>(p.A + ((img * p.H + ih) * p.Wd + iw) * p.Cin + ci));
        } else if (kk + 3 < p.K && (p.lda & 3) == 0) {
          av = __ldg(reinterpret_cast<const float4*>(p.A + m * p.lda + kk));
        } else {
          float t[4] = {0.f, 0.f, 0.f, 0.f};
          for (int i = 0; i < 4; ++i) if (kk + i < p.K) t[i] = __ldg(p.A + m * p.lda + kk + i);
          av = make_float4(t[0], t[1], t[2], t[3]);
        }
      }
    }
    *reinterpret_cast<float4*>(&Zs[lr][lc]) = zv;
    *reinterpret_cast<float4*>(&As[lr][lc]) = av;
    __syncthreads();
#pragma unroll
    for (int r = 0; r < BM; ++r) {
      const float4 zf = *reinterpret_cast<const float4*>(&Zs[r][ty * 4]);
      const float4 af = *reinterpret_cast<const float4*>(&As[r][tx * 4]);
      const float zz[4] = {zf.x, zf.y, zf.z, zf.w}, aa[4] = {af.x, af.y, af.z, af.w};
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(zz[i], aa[j], acc[i][j]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int n = n0 + ty * 4 + i;
    if (n >= p.N) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int k = k0 + tx * 4 + j;
      if (k < p.K) atomicAdd(p.dW + (long long)n * p.K + k, acc[i][j]);
    }
  }
}
void launch_wgrad(WgradP p, int num_sms, cudaStream_t st) {
  const int tn = (p.N + 63) / 64, tk = (p.K + 63) / 64;
  // enough m-splits for ~4 waves of CTAs, at least 64 rows each (256 left the late-stage layers of a 16-image batch,
  // M = 512 rows, at two splits: 192 CTAs walking 16 slabs each)
  long long splits = (4LL * num_sms + tn * tk - 1) / (tn * tk);
  const long long max_splits = (p.M + 63) / 64;
  if (splits > max_splits) splits = max_splits;
  if (splits < 1) splits = 1;
  p.m_chunk = ((p.M + splits - 1) / splits + 15) / 16 * 16;
  splits = (p.M + p.m_chunk - 1) / p.m_chunk;
  wgrad_kernel<<<dim3(tn, tk, (unsigned)splits), 256, 0, st>>>(p);
}

// column sums: db[c] += sum_m dz[m][c]
__global__ void __launch_bounds__(256) colsum_kernel(const float* __restrict__ dz, float* __restrict__ db, long long M, int C, int ld, int rows_per_cta) {
  const int cl = threadIdx.x & 31, rl = threadIdx.x >> 5;
  const int c = blockIdx.x * 32 + cl;
  const long long r0 = (long long)blockIdx.y * rows_per_cta;
  const long long r1 = r0 + rows_per_cta < M ? r0 + rows_per_cta : M;
  float s = 0.f;
  if (c < C)
    for (long long r = r0 + rl; r < r1; r += 8) s += __ldg(dz + r * ld + c);
  __shared__ float ss[8][33];
  ss[rl][cl] = s;
  __syncthreads();
  if (rl == 0 && c < C) {
    float S = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) S += ss[i][cl];
    atomicAdd(db + c, S);
  }
}
void launch_colsum(const float* dz, float* db, long long M, int C, int ld, cudaStream_t st) {
  long long chunks = (M + 511) / 512;
  if (chunks > 512) chunks = 512;
  const int rows = (int)((M + chunks - 1) / chunks);
  colsum_kernel<<<dim3((C + 31) / 32, (unsigned)((M + rows - 1) / rows)), 256, 0, st>>>(dz, db, M, C, ld, rows);
}

// =====================================================================================================================
// depthwise 3x3 backward (NHWC): data gradient (gather) and filter / bias gradient (per-CTA partial sums + atomics)
// =====================================================================================================================
__global__ void __launch_bounds__(256) dw_bwd_data_kernel(const float* __restrict__ dz, const float* __restrict__ w /*[9][C]*/, float* __restrict__ dx,
                                                          int B, int H, int W, int C, int OH, int OW, int stride, int pad_t, int pad_l) {
  const int C4 = C >> 2;
  long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (long long)B * H * W * C4) return;
  const int c = (int)(idx % C4) * 4;
  long long pix = idx / C4;
  const int iw = (int)(pix % W), ih = (int)((pix / W) % H), n = (int)(pix / ((long long)W * H));
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
  for (int kh = 0; kh < 3; ++kh) {
    const int t = ih + pad_t - kh;
    if (t < 0 || t % stride) continue;
    const int oh = t / stride;
    if (oh >= OH) continue;
#pragma unroll
    for (int kw = 0; kw < 3; ++kw) {
      const int u = iw + pad_l - kw;
      if (u < 0 || u % stride) continue;
      const int ow = u / stride;
      if (ow >= OW) continue;
      const float4 g = __ldg(reinterpret_cast<const float4*>(dz + (((long long)n * OH + oh) * OW + ow) * C + c));
      const float4 ww = __ldg(reinterpret_cast<const float4*>(w + (kh * 3 + kw) * C + c));
      acc.x = fmaf(g.x, ww.x, acc.x); acc.y = fmaf(g.y, ww.y, acc.y); acc.z = fmaf(g.z, ww.z, acc.z); acc.w = fmaf(g.w, ww.w, acc.w);
    }
  }
  *reinterpret_cast<float4*>(dx + idx * 4) = acc;
}
// CTA: 32 channels x 8 pixel lanes over a chunk of output pixels; dw[tap][c] += sum dz * x(tap); db[c] += sum dz
__global__ void __launch_bounds__(256) dw_bwd_filter_kernel(const float* __restrict__ dz, const float* __restrict__ x, float* __restrict__ dw, float* __restrict__ db,
                                                            int B, int H, int W, int C, int OH, int OW, int stride, int pad_t, int pad_l, int pix_per_cta) {
  const int cl = threadIdx.x & 31, rl = threadIdx.x >> 5;
  const int c = blockIdx.x * 32 + cl;
  const long long P = (long long)B * OH * OW;
  const long long p0 = (long long)blockIdx.y * pix_per_cta;
  const long long p1 = p0 + pix_per_cta < P ? p0 + pix_per_cta : P;
  float acc[10];
#pragma unroll
  for (int i = 0; i < 10; ++i) acc[i] = 0.f;
  if (c < C)
    for (long long pp = p0 + rl; pp < p1; pp += 8) {
      const int ow = (int)(pp % OW), oh = (int)((pp / OW) % OH);
      const long long n = pp / ((long long)OW * OH);
      const float g = __ldg(dz + pp * C + c);
      acc[9] += g;
#pragma unroll
      for (int kh = 0; kh < 3; ++kh) {
        const int ih = oh * stride - pad_t + kh;
        if (ih < 0 || ih >= H) continue;
#pragma unroll
        for (int kw = 0; kw < 3; ++kw) {
          const int iw = ow * stride - pad_l + kw;
          if (iw < 0 || iw >= W) continue;
          acc[kh * 3 + kw] = fmaf(g, __ldg(x + ((n * H + ih) * W + iw) * C + c), acc[kh * 3 + kw]);
        }
      }
    }
  __shared__ float ss[8][10][33];
#pragma unroll
  for (int i = 0; i < 10; ++i) ss[rl][i][cl] = acc[i];
  __syncthreads();
  if (rl == 0 && c < C) {
#pragma unroll
    for (int i = 0; i < 10; ++i) {
      float S = 0.f;
#pragma unroll
      for (int r = 0; r < 8; ++r) S += ss[r][i][cl];
      if (i < 9) atomicAdd(dw + i * C + c, S);
      else if (db) atomicAdd(db + c, S);
    }
  }
}
void launch_dw_bwd(const float* dz, const float* x, const float* w, float* dx, float* dw, float* db, int B, int H, int W, int C, int OH, int OW,
                   int stride, int pad_t, int pad_l, cudaStream_t st) {
  const long long n = (long long)B * H * W * (C / 4);
  dw_bwd_data_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(dz, w, dx, B, H, W, C, OH, OW, stride, pad_t, pad_l);
  const long long P = (long long)B * OH * OW;
  long long chunks = (P + 255) / 256;
  const long long cgroups = (C + 31) / 32;
  if (cgroups * chunks < 600) chunks = (600 + cgroups - 1) / cgroups;   // small late-stage maps: more pixel chunks, not two long serial walks
  if (chunks > (P + 7) / 8) chunks = (P + 7) / 8;
  if (chunks > 256) chunks = 256;
  if (chunks < 1) chunks = 1;
  const int per = (int)((P + chunks - 1) / chunks);
  dw_bwd_filter_kernel<<<dim3((C + 31) / 32, (unsigned)((P + per - 1) / per)), 256, 0, st>>>(dz, x, dw, db, B, H, W, C, OH, OW, stride, pad_t,
                                                                                             pad_l, per);
}

// =====================================================================================================================
// per-image spatial reductions and broadcasts (squeeze-excite, adaptive 2-D positional encoding)
// =====================================================================================================================
// out[b][c] = scale * sum_q a[b][q][c] * (b2 ? b2[b][q][c] : 1)
__global__ void __launch_bounds__(256) spatial_dot_kernel(const float* __restrict__ a, const float* __restrict__ b2, float* __restrict__ out, int S, int C,
                                                          float scale) {
  const int b = blockIdx.y;
  const int c = blockIdx.x * 256 + threadIdx.x;
  if (c >= C) return;
  const float* ap = a + (long long)b * S * C + c;
  const float* bp = b2 ? b2 + (long long)b * S * C + c : nullptr;
  float s = 0.f;
  for (int q = 0; q < S; ++q) s = bp ? fmaf(__ldg(ap + (long long)q * C), __ldg(bp + (long long)q * C), s) : s + __ldg(ap + (long long)q * C);
  out[(long long)b * C + c] = s * scale;
}
// the same product-sum (b2 != nullptr: the backward pass of the squeeze-excite gate) with the S rows split over four row
// lanes per channel: 4x the CTAs and a quarter of the serial walk (the forward means keep the kernel above and its order)
__global__ void __launch_bounds__(256) spatial_dot4_kernel(const float* __restrict__ a, const float* __restrict__ b2, float* __restrict__ out, int S, int C,
                                                           float scale) {
  __shared__ float part[4][64];
  const int b = blockIdx.y, cl = threadIdx.x & 63, rl = threadIdx.x >> 6;
  const int c = blockIdx.x * 64 + cl;
  float s = 0.f;
  if (c < C) {
    const float* ap = a + (long long)b * S * C + c;
    const float* bp = b2 + (long long)b * S * C + c;
    for (int q = rl; q < S; q += 4) s = fmaf(__ldg(ap + (long long)q * C), __ldg(bp + (long long)q * C), s);
  }
  part[rl][cl] = s;
  __syncthreads();
  if (rl == 0 && c < C) out[(long long)b * C + c] = ((part[0][cl] + part[1][cl]) + (part[2][cl] + part[3][cl])) * scale;
}
void launch_spatial_dot(const float* a, const float* b2, float* out, int B, int S, int C, float scale, cudaStream_t st) {
  if (b2 && S >= 16) {
    spatial_dot4_kernel<<<dim3((C + 63) / 64, B), 256, 0, st>>>(a, b2, out, S, C, scale);
    return;
  }
  spatial_dot_kernel<<<dim3((C + 255) / 256, B), 256, 0, st>>>(a, b2, out, S, C, scale);
}
// out[b][q][c] = x[b][q][c] * g[b][c] (+ add[b][c])   (SE excite; and its backward dy = dout*g + ds/S)
__global__ void __launch_bounds__(256) spatial_scale_kernel(const float* __restrict__ x, const float* __restrict__ g, const float* __restrict__ add,
                                                            float* __restrict__ out, int S, int C, long long n) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int c = (int)(i % C);
  const long long b = i / ((long long)S * C);
  float v = x[i] * g[b * C + c];
  if (add) v += add[b * C + c];
  out[i] = v;
}
void launch_spatial_scale(const float* x, const float* g, const float* add, float* out, int B, int S, int C, cudaStream_t st) {
  const long long n = (long long)B * S * C;
  spatial_scale_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(x, g, add, out, S, C, n);
}

// adaptive 2-D PE apply: out = x + g[b][c] * peh[row][c] + g[b][C + c] * pew[col][c]; with drop.step, dropout on out with
// the mask of the reference's NCHW layout [B, C, h, w]
__global__ void __launch_bounds__(256) pe2d_apply_kernel(const float* __restrict__ x, const float* __restrict__ g, const float* __restrict__ peh,
                                                         const float* __restrict__ pew, float* __restrict__ out, int h, int w, int C, long long n,
                                                         const DropP drop) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int c = (int)(i % C);
  const int q = (int)((i / C) % (h * w));
  const long long b = i / ((long long)h * w * C);
  const float v = x[i] + g[b * 2 * C + c] * __ldg(peh + (q / w) * C + c) + g[b * 2 * C + C + c] * __ldg(pew + (q % w) * C + c);
  out[i] = drop.step ? __fmul_rn(v, drop_factor(drop, (b * C + c) * h * w + q)) : v;
}
void launch_pe2d_apply(const float* x, const float* g, const float* peh, const float* pew, float* out, int B, int h, int w, int C,
                       const DropP& drop, cudaStream_t st) {
  const long long n = (long long)B * h * w * C;
  pe2d_apply_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(x, g, peh, pew, out, h, w, C, n, drop);
}
// dg[b][c] = sum_q dout * peh[row][c];  dg[b][C + c] = sum_q dout * pew[col][c]
__global__ void __launch_bounds__(256) pe2d_bwd_gate_kernel(const float* __restrict__ dout, const float* __restrict__ peh, const float* __restrict__ pew,
                                                            float* __restrict__ dg, int h, int w, int C) {
  const int b = blockIdx.y, c = blockIdx.x * 256 + threadIdx.x;
  if (c >= C) return;
  float sh = 0.f, sw = 0.f;
  for (int q = 0; q < h * w; ++q) {
    const float d = __ldg(dout + ((long long)b * h * w + q) * C + c);
    sh = fmaf(d, __ldg(peh + (q / w) * C + c), sh);
    sw = fmaf(d, __ldg(pew + (q % w) * C + c), sw);
  }
  dg[(long long)b * 2 * C + c] = sh;
  dg[(long long)b * 2 * C + C + c] = sw;
}
void launch_pe2d_bwd_gate(const float* dout, const float* peh, const float* pew, float* dg, int B, int h, int w, int C, cudaStream_t st) {
  pe2d_bwd_gate_kernel<<<dim3((C + 255) / 256, B), 256, 0, st>>>(dout, peh, pew, dg, h, w, C);
}
// x[b][q][c] += add[b][c]
__global__ void __launch_bounds__(256) spatial_add_kernel(float* __restrict__ x, const float* __restrict__ add, int S, int C, long long n, float scale) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  x[i] += scale * add[(i / ((long long)S * C)) * C + (i % C)];
}
void launch_spatial_add(float* x, const float* add, int B, int S, int C, float scale, cudaStream_t st) {
  const long long n = (long long)B * S * C;
  spatial_add_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(x, add, S, C, n, scale);
}

// =====================================================================================================================
// LayerNorm (rows of width C <= 1024, eps 1e-5): forward saving (mean, rstd), backward
// =====================================================================================================================
__global__ void __launch_bounds__(256) ln_fwd_kernel(const float* __restrict__ x, const float* __restrict__ gamma, const float* __restrict__ beta,
                                                     float* __restrict__ y, float* __restrict__ stat /*[M][2]*/, int M, int C) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int m = blockIdx.x * 8 + warp;
  if (m >= M) return;
  const float* xp = x + (long long)m * C;
  float s = 0.f;
  for (int c = lane; c < C; c += 32) s += xp[c];
  const float mean = warp_sum(s) / (float)C;
  float q = 0.f;
  for (int c = lane; c < C; c += 32) { const float d = xp[c] - mean; q = fmaf(d, d, q); }
  const float rstd = rsqrtf(warp_sum(q) / (float)C + 1e-5f);
  for (int c = lane; c < C; c += 32) y[(long long)m * C + c] = (xp[c] - mean) * rstd * __ldg(gamma + c) + __ldg(beta + c);
  if (lane == 0) { stat[2 * m] = mean; stat[2 * m + 1] = rstd; }
}
void launch_ln_fwd(const float* x, const float* gamma, const float* beta, float* y, float* stat, int M, int C, cudaStream_t st) {
  ln_fwd_kernel<<<(M + 7) / 8, 256, 0, st>>>(x, gamma, beta, y, stat, M, C);
}
// dx = rstd * (dyg - mean(dyg) - xhat * mean(dyg * xhat)), dyg = dy * gamma; dgamma += sum dy*xhat; dbeta += sum dy
__global__ void __launch_bounds__(256) ln_bwd_kernel(const float* __restrict__ dy, const float* __restrict__ x, const float* __restrict__ stat,
                                                     const float* __restrict__ gamma, float* __restrict__ dx, float* __restrict__ dgamma,
                                                     float* __restrict__ dbeta, int M, int C, int rows_per_cta) {
  extern __shared__ float sm[];   // [2][C] partial dgamma / dbeta of this CTA
  float* sg = sm;
  float* sb = sm + C;
  for (int c = threadIdx.x; c < 2 * C; c += 256) sm[c] = 0.f;
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int r0 = blockIdx.x * rows_per_cta, r1 = min(M, r0 + rows_per_cta);
  for (int m = r0 + warp; m < r1; m += 8) {
    const float mean = stat[2 * m], rstd = stat[2 * m + 1];
    const float* xp = x + (long long)m * C;
    const float* dp = dy + (long long)m * C;
    float s1 = 0.f, s2 = 0.f;
    for (int c = lane; c < C; c += 32) {
      const float g = dp[c] * __ldg(gamma + c), xh = (xp[c] - mean) * rstd;
      s1 += g;
      s2 = fmaf(g, xh, s2);
    }
    s1 = warp_sum(s1) / (float)C;
    s2 = warp_sum(s2) / (float)C;
    for (int c = lane; c < C; c += 32) {
      const float xh = (xp[c] - mean) * rstd;
      dx[(long long)m * C + c] = rstd * (dp[c] * __ldg(gamma + c) - s1 - xh * s2);
      atomicAdd(sg + c, dp[c] * xh);
      atomicAdd(sb + c, dp[c]);
    }
  }
  __syncthreads();
  for (int c = threadIdx.x; c < C; c += 256) {
    atomicAdd(dgamma + c, sg[c]);
    atomicAdd(dbeta + c, sb[c]);
  }
}
void launch_ln_bwd(const float* dy, const float* x, const float* stat, const float* gamma, float* dx, float* dgamma, float* dbeta, int M, int C,
                   cudaStream_t st) {
  int ctas = (M + 15) / 16;   // two rows per warp: the 512-row LayerNorms of a 16-image batch used 8 CTAs
  if (ctas > 592) ctas = 592;
  const int rows = (M + ctas - 1) / ctas;
  ln_bwd_kernel<<<(M + rows - 1) / rows, 256, 2 * C * sizeof(float), st>>>(dy, x, stat, gamma, dx, dgamma, dbeta, M, C, rows);
}

// =====================================================================================================================
// multi-head attention backward (ScaledDotProductAttention, EfficientSATRN.py:164-172): one CTA per (batch, head);
// probabilities are recomputed from q, k; dk / dv accumulate in shared memory over the queries.
// mask: causal (key j <= query i) and / or key padding (key_mask[b][j] != 0 -> masked), as in the forward kernels.
// =====================================================================================================================
__global__ void __launch_bounds__(256) attn_bwd_kernel(const AttnBwdP p) {
  extern __shared__ float sm[];
  const int HD = p.HD, Lk = p.Lk, Lq = p.Lq;
  float* sk = sm;                    // [Lk][HD+1]
  float* sv = sk + Lk * (HD + 1);
  float* sdk = sv + Lk * (HD + 1);
  float* sdv = sdk + Lk * (HD + 1);
  float* sp = sdv + Lk * (HD + 1);   // [8 warps][Lk] probabilities / ds
  const int b = blockIdx.x / p.heads, hh = blockIdx.x % p.heads;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int i = threadIdx.x; i < Lk * HD; i += 256) {
    const int j = i / HD, d = i % HD;
    sk[j * (HD + 1) + d] = p.k[((long long)b * Lk + j) * p.ldk + hh * HD + d];
    sv[j * (HD + 1) + d] = p.v[((long long)b * Lk + j) * p.ldv + hh * HD + d];
    sdk[j * (HD + 1) + d] = 0.f;
    sdv[j * (HD + 1) + d] = 0.f;
  }
  __syncthreads();
  const float inv_t = 1.f / p.temperature;
  float* pw = sp + warp * Lk;
  for (int i = warp; i < Lq; i += 8) {
    const float* qp = p.q + ((long long)b * Lq + i) * p.ldq + hh * HD;
    const float* dop = p.dout + ((long long)b * Lq + i) * p.ldo + hh * HD;
    // scores
    float mx = -INFINITY;
    for (int j = lane; j < Lk; j += 32) {
      bool masked = (p.causal && j > i) || (p.key_mask && p.key_mask[(long long)b * Lk + j]);
      float s = -INFINITY;
      if (!masked) {
        s = 0.f;
        for (int d = 0; d < HD; ++d) s = fmaf(qp[d], sk[j * (HD + 1) + d], s);
        s *= inv_t;
      }
      pw[j] = s;
      mx = fmaxf(mx, s);
    }
    mx = warp_max(mx);
    float sum = 0.f;
    for (int j = lane; j < Lk; j += 32) {
      const float e = pw[j] == -INFINITY ? 0.f : expf(pw[j] - mx);
      pw[j] = e;
      sum += e;
    }
    sum = warp_sum(sum);
    const float inv = 1.f / sum;
    // dp_j = dout . v_j ; delta = sum_j p_j dp_j
    float delta = 0.f;
    float dpj[8];   // Lk <= 256
    int cnt = 0;
    for (int j = lane; j < Lk; j += 32, ++cnt) {
      const float pj = pw[j] * inv;
      // dropout on the probabilities: the forward multiplied V by P.M.s, so dP = (dout . v_j) M.s and dv_j += P M.s dout
      const float mj = p.drop.step ? drop_factor(p.drop, (((long long)b * p.heads + hh) * Lq + i) * Lk + j) : 1.f;
      float dp = 0.f;
      for (int d = 0; d < HD; ++d) dp = fmaf(dop[d], sv[j * (HD + 1) + d], dp);
      if (p.drop.step) dp = __fmul_rn(dp, mj);
      dpj[cnt] = dp;
      delta = fmaf(pj, dp, delta);
      // dv_j += p_j * dout
      const float pv = p.drop.step ? __fmul_rn(pj, mj) : pj;
      for (int d = 0; d < HD; ++d) atomicAdd(&sdv[j * (HD + 1) + d], pv * dop[d]);
    }
    delta = warp_sum(delta);
    cnt = 0;
    for (int j = lane; j < Lk; j += 32, ++cnt) {
      const float pj = pw[j] * inv;
      const float ds = pj * (dpj[cnt] - delta) * inv_t;
      pw[j] = ds;
      for (int d = 0; d < HD; ++d) atomicAdd(&sdk[j * (HD + 1) + d], ds * qp[d]);
    }
    __syncwarp();
    // dq_i = sum_j ds_j k_j
    for (int d = lane; d < HD; d += 32) {
      float s = 0.f;
      for (int j = 0; j < Lk; ++j) s = fmaf(pw[j], sk[j * (HD + 1) + d], s);
      p.dq[((long long)b * Lq + i) * p.lddq + hh * HD + d] = s;
    }
    __syncwarp();
  }
  __syncthreads();
  for (int i = threadIdx.x; i < Lk * HD; i += 256) {
    const int j = i / HD, d = i % HD;
    float* dk = p.dk + ((long long)b * Lk + j) * p.lddk + hh * HD + d;
    float* dv = p.dv + ((long long)b * Lk + j) * p.lddv + hh * HD + d;
    if (p.accumulate_kv) { *dk += sdk[j * (HD + 1) + d]; *dv += sdv[j * (HD + 1) + d]; }
    else { *dk = sdk[j * (HD + 1) + d]; *dv = sdv[j * (HD + 1) + d]; }
  }
}
// The same backward pass with the queries split over CTAs: grid (batch x head, chunks of ATT_QB queries).  A CTA keeps the
// head's K and V, recomputes the probabilities P and the score gradients dS of its query rows into shared memory (one
// warp per row, writing dq on the way), then reduces dV = P^T dO and dK = dS^T Q over ITS rows with one thread per
// (key, dim) -- no shared-memory atomics -- and adds the result to global dk / dv (zeroed by the launcher unless they
// accumulate).  One CTA per (batch, head) walked 231 x 231 x 32 x 2 shared atomics serially: 625 us per launch.
constexpr int ATT_QB = 16;
__global__ void __launch_bounds__(256) attn_bwd_split_kernel(const AttnBwdP p) {
  extern __shared__ float sm[];
  const int HD = p.HD, Lk = p.Lk, Lq = p.Lq;
  float* sk = sm;                       // [Lk][HD+1]
  float* sv = sk + Lk * (HD + 1);       // [Lk][HD+1]
  float* sP = sv + Lk * (HD + 1);       // [ATT_QB][Lk]  probabilities
  float* sS = sP + ATT_QB * Lk;         // [ATT_QB][Lk]  dS
  float* sq = sS + ATT_QB * Lk;         // [ATT_QB][HD]
  float* sdo = sq + ATT_QB * HD;        // [ATT_QB][HD]
  const int b = blockIdx.x / p.heads, hh = blockIdx.x % p.heads;
  const int i0 = blockIdx.y * ATT_QB;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int i = threadIdx.x; i < Lk * HD; i += 256) {
    const int j = i / HD, d = i % HD;
    sk[j * (HD + 1) + d] = p.k[((long long)b * Lk + j) * p.ldk + hh * HD + d];
    sv[j * (HD + 1) + d] = p.v[((long long)b * Lk + j) * p.ldv + hh * HD + d];
  }
  for (int i = threadIdx.x; i < ATT_QB * HD; i += 256) {
    const int r = i / HD, d = i % HD;
    const bool ok = i0 + r < Lq;
    sq[i] = ok ? p.q[((long long)b * Lq + i0 + r) * p.ldq + hh * HD + d] : 0.f;
    sdo[i] = ok ? p.dout[((long long)b * Lq + i0 + r) * p.ldo + hh * HD + d] : 0.f;
  }
  __syncthreads();
  const float inv_t = 1.f / p.temperature;
  for (int r = warp; r < ATT_QB; r += 8) {
    const int i = i0 + r;
    float* pw = sP + r * Lk;
    float* dsw = sS + r * Lk;
    if (i >= Lq) {
      for (int j = lane; j < Lk; j += 32) { pw[j] = 0.f; dsw[j] = 0.f; }
      continue;
    }
    const float* qp = sq + r * HD;
    const float* dop = sdo + r * HD;
    float mx = -INFINITY;
    for (int j = lane; j < Lk; j += 32) {
      const bool masked = (p.causal && j > i) || (p.key_mask && p.key_mask[(long long)b * Lk + j]);
      float sc = -INFINITY;
      if (!masked) {
        sc = 0.f;
        for (int d = 0; d < HD; ++d) sc = fmaf(qp[d], sk[j * (HD + 1) + d], sc);
        sc *= inv_t;
      }
      pw[j] = sc;
      mx = fmaxf(mx, sc);
    }
    mx = warp_max(mx);
    float sum = 0.f;
    for (int j = lane; j < Lk; j += 32) {
      const float e = pw[j] == -INFINITY ? 0.f : expf(pw[j] - mx);
      pw[j] = e;
      sum += e;
    }
    sum = warp_sum(sum);
    const float inv = 1.f / sum;
    float delta = 0.f;
    const long long erow = (((long long)b * p.heads + hh) * Lq + i) * Lk;   // dropout mask row (logical [B, heads, Lq, Lk])
    for (int j = lane; j < Lk; j += 32) {
      const float pj = pw[j] * inv;
      float dp = 0.f;
      for (int d = 0; d < HD; ++d) dp = fmaf(dop[d], sv[j * (HD + 1) + d], dp);
      if (p.drop.step) dp = __fmul_rn(dp, drop_factor(p.drop, erow + j));   // dP = (dO V^T) M.s
      pw[j] = pj;
      dsw[j] = dp;
      delta = fmaf(pj, dp, delta);
    }
    delta = warp_sum(delta);
    for (int j = lane; j < Lk; j += 32) dsw[j] = pw[j] * (dsw[j] - delta) * inv_t;
    if (p.drop.step)   // dV below takes the probabilities the forward multiplied V by: P.M.s
      for (int j = lane; j < Lk; j += 32) pw[j] = __fmul_rn(pw[j], drop_factor(p.drop, erow + j));
    __syncwarp();
    for (int d = lane; d < HD; d += 32) {   // dq_i = sum_j ds_j k_j
      float acc = 0.f;
      for (int j = 0; j < Lk; ++j) acc = fmaf(dsw[j], sk[j * (HD + 1) + d], acc);
      p.dq[((long long)b * Lq + i) * p.lddq + hh * HD + d] = acc;
    }
  }
  __syncthreads();
  // dV[j][d] = sum_r P[r][j] dO[r][d],  dK[j][d] = sum_r dS[r][j] Q[r][d] over this CTA's rows
  for (int j = warp; j < Lk; j += 8) {
    for (int d = lane; d < HD; d += 32) {
      float av = 0.f, ak = 0.f;
#pragma unroll 8
      for (int r = 0; r < ATT_QB; ++r) {
        av = fmaf(sP[r * Lk + j], sdo[r * HD + d], av);
        ak = fmaf(sS[r * Lk + j], sq[r * HD + d], ak);
      }
      atomicAdd(p.dv + ((long long)b * Lk + j) * p.lddv + hh * HD + d, av);
      atomicAdd(p.dk + ((long long)b * Lk + j) * p.lddk + hh * HD + d, ak);
    }
  }
}

int launch_attn_bwd(const AttnBwdP& p, int B, cudaStream_t st) {
  if (p.Lk > 256) return (int)cudaErrorInvalidValue;
  const size_t smem2 = ((size_t)2 * p.Lk * (p.HD + 1) + 2 * ATT_QB * p.Lk + 2 * ATT_QB * p.HD) * sizeof(float);
  if (smem2 <= 200 * 1024) {
    static SmemOptIn opt2;
    cudaError_t e = opt2.ensure(attn_bwd_split_kernel, smem2);
    if (e != cudaSuccess) return (int)e;
    if (!p.accumulate_kv) {   // the CTAs of a (batch, head) add their partial dk / dv
      const size_t w = (size_t)p.heads * p.HD * sizeof(float);
      e = cudaMemset2DAsync(p.dk, (size_t)p.lddk * sizeof(float), 0, w, (size_t)B * p.Lk, st);
      if (e != cudaSuccess) return (int)e;
      e = cudaMemset2DAsync(p.dv, (size_t)p.lddv * sizeof(float), 0, w, (size_t)B * p.Lk, st);
      if (e != cudaSuccess) return (int)e;
    }
    attn_bwd_split_kernel<<<dim3(B * p.heads, (p.Lq + ATT_QB - 1) / ATT_QB), 256, smem2, st>>>(p);
    return 0;
  }
  const size_t smem = ((size_t)4 * p.Lk * (p.HD + 1) + 8 * p.Lk) * sizeof(float);
  static SmemOptIn opt;
  cudaError_t e = opt.ensure(attn_bwd_kernel, smem);
  if (e != cudaSuccess) return (int)e;
  attn_bwd_kernel<<<B * p.heads, 256, smem, st>>>(p);
  return 0;
}

// =====================================================================================================================
// embedding backward, cross-entropy (ignore_index) forward + backward
// =====================================================================================================================
// dE[tok[m]][:] += scale * dx[m][:]
__global__ void __launch_bounds__(256) embed_bwd_kernel(const long long* __restrict__ tok, const float* __restrict__ dx, float* __restrict__ dE, int M, int D,
                                                        float scale) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (long long)M * D) return;
  const int m = (int)(i / D), d = (int)(i % D);
  atomicAdd(dE + tok[m] * D + d, scale * dx[i]);
}
void launch_embed_bwd(const long long* tok, const float* dx, float* dE, int M, int D, float scale, cudaStream_t st) {
  const long long n = (long long)M * D;
  embed_bwd_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(tok, dx, dE, M, D, scale);
}

// targets[m] = expected[b][l+1]; one warp per row: nll, dlogits = (softmax - onehot) / n_valid (0 for ignored rows).
// pass 0 (count): n_valid; pass 1: loss sum and gradients.
__global__ void __launch_bounds__(256) ce_count_kernel(const long long* __restrict__ expected, int B, int L, int pad, float* __restrict__ out2) {
  int n = 0;
  for (int i = threadIdx.x; i < B * L; i += 256) n += expected[(long long)(i / L) * (L + 1) + (i % L) + 1] != pad;
  __shared__ int s[256];
  s[threadIdx.x] = n;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) { if (threadIdx.x < o) s[threadIdx.x] += s[threadIdx.x + o]; __syncthreads(); }
  if (threadIdx.x == 0) { out2[0] = 0.f; out2[1] = (float)s[0]; }
}
__global__ void __launch_bounds__(256) ce_kernel(const float* __restrict__ logits, const long long* __restrict__ expected, float* __restrict__ dlogits,
                                                 float* __restrict__ out2 /*[0] loss (mean), [1] n_valid*/, int B, int L, int V, int pad) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int m = blockIdx.x * 8 + warp;
  if (m >= B * L) return;
  const long long tgt = expected[(long long)(m / L) * (L + 1) + (m % L) + 1];
  const float* lp = logits + (long long)m * V;
  float* dp = dlogits + (long long)m * V;
  const float nv = out2[1];
  if (tgt == pad) {
    for (int v = lane; v < V; v += 32) dp[v] = 0.f;
    return;
  }
  float mx = -INFINITY;
  for (int v = lane; v < V; v += 32) mx = fmaxf(mx, lp[v]);
  mx = warp_max(mx);
  float s = 0.f;
  for (int v = lane; v < V; v += 32) s += expf(lp[v] - mx);
  s = warp_sum(s);
  const float lse = mx + logf(s);
  const float invn = 1.f / nv;
  for (int v = lane; v < V; v += 32) dp[v] = (expf(lp[v] - lse) - (v == tgt ? 1.f : 0.f)) * invn;
  if (lane == 0) atomicAdd(out2, (lse - lp[tgt]) * invn);
}
void launch_cross_entropy(const float* logits, const long long* expected, float* dlogits, float* out2, int B, int L, int V, int pad, cudaStream_t st) {
  ce_count_kernel<<<1, 256, 0, st>>>(expected, B, L, pad, out2);
  ce_kernel<<<(B * L + 7) / 8, 256, 0, st>>>(logits, expected, dlogits, out2, B, L, V, pad);
}

// stem convolution (3x3, stride 2, padding 0, NCHW image -> NHWC): filter gradient dW[co][ci][kh][kw]
__global__ void __launch_bounds__(256) stem_wgrad_kernel(const float* __restrict__ dz, const float* __restrict__ img, float* __restrict__ dw, int B, int Cin,
                                                         int H, int W, int OH, int OW, int Cout, int pix_per_cta) {
  extern __shared__ float sm[];   // [Cout * Cin * 9]
  const int nW = Cout * Cin * 9;
  for (int i = threadIdx.x; i < nW; i += 256) sm[i] = 0.f;
  __syncthreads();
  const long long P = (long long)B * OH * OW;
  const long long p0 = (long long)blockIdx.x * pix_per_cta;
  const long long p1 = p0 + pix_per_cta < P ? p0 + pix_per_cta : P;
  // thread -> (co, pixel lane): Cout <= 32
  const int co = threadIdx.x % 32, pl = threadIdx.x / 32;
  if (co < Cout) {
    for (int ci = 0; ci < Cin; ++ci) {
      float acc[9];
#pragma unroll
      for (int t = 0; t < 9; ++t) acc[t] = 0.f;
      for (long long pp = p0 + pl; pp < p1; pp += 8) {
        const int ow = (int)(pp % OW), oh = (int)((pp / OW) % OH);
        const long long n = pp / ((long long)OW * OH);
        const float g = __ldg(dz + pp * Cout + co);
        const float* ip = img + ((n * Cin + ci) * H + oh * 2) * W + ow * 2;
#pragma unroll
        for (int kh = 0; kh < 3; ++kh)
#pragma unroll
          for (int kw = 0; kw < 3; ++kw) acc[kh * 3 + kw] = fmaf(g, __ldg(ip + kh * W + kw), acc[kh * 3 + kw]);
      }
#pragma unroll
      for (int t = 0; t < 9; ++t) atomicAdd(&sm[(co * Cin + ci) * 9 + t], acc[t]);
    }
  }
  __syncthreads();
  for (int i = threadIdx.x; i < nW; i += 256) atomicAdd(dw + i, sm[i]);
}
// Weight gradient of a 3 x 3 convolution that reads the NCHW input image (any stride / padding, Cout a divisor of 256):
// LiteSATRN's conv0 (networks/LiteSATRN.py:24-26: 1 -> 128 channels, stride 1, padding 1).  dw [Cout][Cin][3][3].
__global__ void __launch_bounds__(256) image_conv_wgrad_kernel(const float* __restrict__ dz, const float* __restrict__ img, float* __restrict__ dw,
                                                               int B, int Cin, int H, int W, int OH, int OW, int Cout, int stride, int pad,
                                                               int pix_per_cta) {
  extern __shared__ float sm[];   // [Cout * Cin * 9]
  const int nW = Cout * Cin * 9;
  for (int i = threadIdx.x; i < nW; i += 256) sm[i] = 0.f;
  __syncthreads();
  const long long P = (long long)B * OH * OW;
  const long long p0 = (long long)blockIdx.x * pix_per_cta;
  const long long p1 = p0 + pix_per_cta < P ? p0 + pix_per_cta : P;
  const int lanes = 256 / Cout, co = threadIdx.x % Cout, pl = threadIdx.x / Cout;
  for (int ci = 0; ci < Cin; ++ci) {
    float acc[9];
#pragma unroll
    for (int t = 0; t < 9; ++t) acc[t] = 0.f;
    for (long long pp = p0 + pl; pp < p1; pp += lanes) {
      const int ow = (int)(pp % OW), oh = (int)((pp / OW) % OH);
      const long long n = pp / ((long long)OW * OH);
      const float g = __ldg(dz + pp * Cout + co);
      const float* ip = img + (n * Cin + ci) * (long long)H * W;
#pragma unroll
      for (int kh = 0; kh < 3; ++kh) {
        const int ih = oh * stride - pad + kh;
#pragma unroll
        for (int kw = 0; kw < 3; ++kw) {
          const int iw = ow * stride - pad + kw;
          if (ih >= 0 && ih < H && iw >= 0 && iw < W) acc[kh * 3 + kw] = fmaf(g, __ldg(ip + (long long)ih * W + iw), acc[kh * 3 + kw]);
        }
      }
    }
#pragma unroll
    for (int t = 0; t < 9; ++t) atomicAdd(&sm[(co * Cin + ci) * 9 + t], acc[t]);
  }
  __syncthreads();
  for (int i = threadIdx.x; i < nW; i += 256) atomicAdd(dw + i, sm[i]);
}
int launch_image_conv_wgrad(const float* dz, const float* img, float* dw, int B, int Cin, int H, int W, int OH, int OW, int Cout, int stride,
                            int pad, cudaStream_t st) {
  if (Cout <= 0 || Cout > 256 || 256 % Cout != 0 || (size_t)Cout * Cin * 9 * sizeof(float) > 48 * 1024) return 1;
  const long long P = (long long)B * OH * OW;
  const int per = 2048;
  image_conv_wgrad_kernel<<<(unsigned)((P + per - 1) / per), 256, (size_t)Cout * Cin * 9 * sizeof(float), st>>>(dz, img, dw, B, Cin, H, W, OH, OW,
                                                                                                              Cout, stride, pad, per);
  return 0;
}

// 2 x 2 / stride 2 max pooling over NHWC (nn.MaxPool2d(2, 2), LiteSATRN.py:29) and its backward pass.  The gradient goes
// to the FIRST maximum of the window in (row, column) scan order, like ATen's max_pool2d_with_indices (after a ReLU whole
// windows of zeros are common); every input element belongs to exactly one window (H, W even), so dx is written, not
// accumulated.
__global__ void __launch_bounds__(256) maxpool2_fwd_kernel(const float* __restrict__ x, float* __restrict__ y, int B, int H, int W, int C) {
  const int OH = H / 2, OW = W / 2, C4 = C / 4;
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (long long)B * OH * OW * C4) return;
  const int c = (int)(i % C4) * 4;
  long long pix = i / C4;
  const int ow = (int)(pix % OW), oh = (int)((pix / OW) % OH), n = (int)(pix / ((long long)OW * OH));
  const float* xp = x + (((long long)n * H + 2 * oh) * W + 2 * ow) * C + c;
  const float4 a = *reinterpret_cast<const float4*>(xp), b = *reinterpret_cast<const float4*>(xp + C);
  const float4 d = *reinterpret_cast<const float4*>(xp + (long long)W * C), e = *reinterpret_cast<const float4*>(xp + (long long)W * C + C);
  float4 o;
  o.x = fmaxf(fmaxf(a.x, b.x), fmaxf(d.x, e.x)); o.y = fmaxf(fmaxf(a.y, b.y), fmaxf(d.y, e.y));
  o.z = fmaxf(fmaxf(a.z, b.z), fmaxf(d.z, e.z)); o.w = fmaxf(fmaxf(a.w, b.w), fmaxf(d.w, e.w));
  *reinterpret_cast<float4*>(y + i * 4) = o;
}
void launch_maxpool2_fwd(const float* x, float* y, int B, int H, int W, int C, cudaStream_t st) {
  const long long n = (long long)B * (H / 2) * (W / 2) * (C / 4);
  maxpool2_fwd_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(x, y, B, H, W, C);
}
__global__ void __launch_bounds__(256) maxpool2_bwd_kernel(const float* __restrict__ x, const float* __restrict__ dy, float* __restrict__ dx, int B,
                                                           int H, int W, int C) {
  const int OH = H / 2, OW = W / 2;
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (long long)B * OH * OW * C) return;
  const int c = (int)(i % C);
  long long pix = i / C;
  const int ow = (int)(pix % OW), oh = (int)((pix / OW) % OH), n = (int)(pix / ((long long)OW * OH));
  const long long base = (((long long)n * H + 2 * oh) * W + 2 * ow) * C + c;
  const long long off[4] = {0, C, (long long)W * C, (long long)W * C + C};
  int best = 0;
  float bv = x[base];
#pragma unroll
  for (int k = 1; k < 4; ++k) {
    const float v = x[base + off[k]];
    if (v > bv) { bv = v; best = k; }
  }
  const float g = dy[i];
#pragma unroll
  for (int k = 0; k < 4; ++k) dx[base + off[k]] = k == best ? g : 0.f;
}
void launch_maxpool2_bwd(const float* x, const float* dy, float* dx, int B, int H, int W, int C, cudaStream_t st) {
  const long long n = (long long)B * (H / 2) * (W / 2) * C;
  maxpool2_bwd_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(x, dy, dx, B, H, W, C);
}

void launch_stem_wgrad(const float* dz, const float* img, float* dw, int B, int Cin, int H, int W, int OH, int OW, int Cout, cudaStream_t st) {
  const long long P = (long long)B * OH * OW;
  const int per = 2048;
  stem_wgrad_kernel<<<(unsigned)((P + per - 1) / per), 256, (size_t)Cout * Cin * 9 * sizeof(float), st>>>(dz, img, dw, B, Cin, H, W, OH, OW, Cout, per);
}

// =====================================================================================================================
// optimiser: global gradient norm, clip_grad_norm_(max_norm) and AdamW (torch.optim.AdamW defaults: betas (0.9, 0.999),
// eps 1e-8, decoupled weight decay p *= 1 - lr*wd)
// =====================================================================================================================
__global__ void __launch_bounds__(256) sumsq_kernel(const float* __restrict__ g, long long n, double* __restrict__ out) {
  double s = 0;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const double v = g[i];
    s += v * v;
  }
  s = warp_sum_d(s);
  __shared__ double ws[8];
  if ((threadIdx.x & 31) == 0) ws[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0;
    for (int i = 0; i < 8; ++i) t += ws[i];
    atomicAdd(out, t);
  }
}
void launch_sumsq(const float* g, long long n, double* out, cudaStream_t st) {
  cudaMemsetAsync(out, 0, sizeof(double), st);
  sumsq_kernel<<<592, 256, 0, st>>>(g, n, out);
}
// sumsq[0] holds the squared norm of the (already averaged) gradient; writes the norm to norm_out
__global__ void __launch_bounds__(256) adamw_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m, float* __restrict__ v,
                                                    const double* __restrict__ sumsq, float* __restrict__ norm_out, long long n, float lr, float wd,
                                                    float beta1, float beta2, float eps, float bc1, float bc2, float max_norm, float grad_scale) {
  const float norm = (float)sqrt(*sumsq) * grad_scale;
  if (blockIdx.x == 0 && threadIdx.x == 0 && norm_out) *norm_out = norm;
  float clip = max_norm > 0.f ? max_norm / (norm + 1e-6f) : 1.f;   // torch.nn.utils.clip_grad_norm_
  if (clip > 1.f) clip = 1.f;
  const float gs = clip * grad_scale;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const float gg = g[i] * gs;
    float pp = p[i] * (1.f - lr * wd);
    const float mm = beta1 * m[i] + (1.f - beta1) * gg;
    const float vv = beta2 * v[i] + (1.f - beta2) * gg * gg;
    m[i] = mm;
    v[i] = vv;
    const float denom = sqrtf(vv) / sqrtf(bc2) + eps;
    pp -= (lr / bc1) * (mm / denom);
    p[i] = pp;
  }
}
void launch_adamw(float* p, const float* g, float* m, float* v, const double* sumsq, float* norm_out, long long n, float lr, float wd, int step,
                  float max_norm, float grad_scale, cudaStream_t st) {
  const float b1 = 0.9f, b2 = 0.999f;
  const float bc1 = 1.f - powf(b1, (float)step), bc2 = 1.f - powf(b2, (float)step);
  adamw_kernel<<<592, 256, 0, st>>>(p, g, m, v, sumsq, norm_out, n, lr, wd, b1, b2, 1e-8f, bc1, bc2, max_norm, grad_scale);
}

// row softmax-free helpers for the teacher-forced decoder: out[m][:] = in[m][:] (+ bias) with optional ReLU -- not needed:
// linear layers go through launch_igemm_f32 (bias = shift, act in the epilogue).

}  // namespace frx
