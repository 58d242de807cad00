// kernels_f32.cu -- fp32 (no TF32) kernel set of the frx hot path.
//
// This is the bit-faithful mode (BASELINE.json: "decoded token IDs must be
// bit-exact in fp32 mode"): every contraction accumulates in fp32 FFMA in a
// fixed order, so results are deterministic run to run.  The bf16 tensor-core
// kernels (kernels_bf16*.cu) replace the dense contractions in bf16 mode.
//
// Reference lines cited are in /root/reference/networks/EfficientSATRN.py.
#include "common.cuh"
#include "kernels.h"

namespace frx {

// ===========================================================================
// 1. Stem: conv3x3 stride 2 padding 0 (1..3 -> Cout) + BN + SiLU   (:67-73,:82-83)
//    input NCHW fp32, output NHWC fp32.  HBM-bound, one thread per output value.
// ===========================================================================
__global__ void __launch_bounds__(256) stem_conv_kernel(const float* __restrict__ in,
                                                        const float* __restrict__ w,   // [Cout][Cin][3][3]
                                                        const float* __restrict__ scale,
                                                        const float* __restrict__ shift,
                                                        float* __restrict__ out, int B, int Cin, int H,
                                                        int W, int OH, int OW, int Cout, int stride, int pad,
                                                        int act) {
  extern __shared__ float ws[];  // Cout*Cin*9 + 2*Cout
  for (int i = threadIdx.x; i < Cout * Cin * 9; i += blockDim.x) ws[i] = w[i];
  float* ssc = ws + Cout * Cin * 9;
  float* ssh = ssc + Cout;
  for (int i = threadIdx.x; i < Cout; i += blockDim.x) { ssc[i] = scale[i]; ssh[i] = shift[i]; }
  __syncthreads();
  long long total = (long long)B * OH * OW * Cout;
  long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= total) return;
  int co = (int)(idx % Cout);
  long long pix = idx / Cout;
  int ow = (int)(pix % OW);
  int oh = (int)((pix / OW) % OH);
  int n = (int)(pix / ((long long)OW * OH));
  float acc = 0.f;
  for (int ci = 0; ci < Cin; ++ci) {
    const float* ip = in + ((long long)n * Cin + ci) * H * W;
    const float* wp = ws + (co * Cin + ci) * 9;
#pragma unroll
    for (int kh = 0; kh < 3; ++kh) {
      const int ih = oh * stride - pad + kh;
      if (ih < 0 || ih >= H) continue;
#pragma unroll
      for (int kw = 0; kw < 3; ++kw) {
        const int iw = ow * stride - pad + kw;
        if (iw < 0 || iw >= W) continue;
        acc = fmaf(__ldg(ip + (long long)ih * W + iw), wp[kh * 3 + kw], acc);
      }
    }
  }
  out[idx] = act_apply(acc * ssc[co] + ssh[co], act);
}

void launch_stem_conv(const float* in, const float* w, const float* scale, const float* shift,
                      float* out, int B, int Cin, int H, int W, int OH, int OW, int Cout,
                      cudaStream_t st) {
  launch_direct_conv3x3(in, w, scale, shift, out, B, Cin, H, W, OH, OW, Cout, 2, 0, ACT_SILU, st);
}

// Direct 3x3 convolution from an NCHW fp32 image (few input channels) to NHWC fp32:
// EfficientSATRN stem (stride 2, padding 0, SiLU) and LiteSATRN conv0 (stride 1, padding 1, ReLU).
void launch_direct_conv3x3(const float* in, const float* w, const float* scale, const float* shift, float* out, int B,
                           int Cin, int H, int W, int OH, int OW, int Cout, int stride, int pad, int act,
                           cudaStream_t st) {
  long long total = (long long)B * OH * OW * Cout;
  int smem = (Cout * Cin * 9 + 2 * Cout) * sizeof(float);
  stem_conv_kernel<<<(unsigned)((total + 255) / 256), 256, smem, st>>>(in, w, scale, shift, out, B, Cin,
                                                                      H, W, OH, OW, Cout, stride, pad, act);
}

// ===========================================================================
// 2. Implicit-GEMM convolution / dense GEMM, fp32 SIMT.
//    C[M,N] = epi( A[M,K] * W[N,K]^T ), A gathered from NHWC for 3x3 convs.
//    256 threads, BK = 16, register prefetch of the next K slab.
// ===========================================================================
template <int BM, int BN, int TM, int TN>
__global__ void __launch_bounds__(256) igemm_f32_kernel(const GemmP p) {
  constexpr int BK = 16;
  constexpr int AL = BM * 4 / 256;  // float4 loads of A per thread per slab
  constexpr int BL = BN * 4 / 256 > 0 ? BN * 4 / 256 : 1;
  constexpr bool B_PARTIAL = (BN * 4 < 256);
  static_assert((BM / TM) * (BN / TN) == 256, "tile/thread mismatch");
  __shared__ __align__(16) float As[BK][BM + 4];
  __shared__ __align__(16) float Bs[BK][BN + 4];

  const int tid = threadIdx.x;
  const int m0 = blockIdx.x * BM, n0 = blockIdx.y * BN;

  // ---- per-thread loader coordinates -------------------------------------
  int a_row[AL], a_kq[AL];
  const float* a_base[AL];  // dense: row pointer; conv: image base pointer
  int a_ih0[AL], a_iw0[AL];
  bool a_ok[AL];
  const float* a_gate[AL];
#pragma unroll
  for (int i = 0; i < AL; ++i) {
    int id = tid + i * 256;
    a_row[i] = id >> 2;
    a_kq[i] = (id & 3) * 4;
    int m = m0 + a_row[i];
    a_ok[i] = m < p.M;
    a_gate[i] = nullptr;
    a_ih0[i] = a_iw0[i] = 0;
    if (!a_ok[i]) { a_base[i] = p.A; continue; }
    if (p.conv) {
      int ow = m % p.OW;
      int t = m / p.OW;
      int oh = t % p.OH;
      int n = t / p.OH;
      a_base[i] = p.A + (long long)n * p.H * p.Wd * p.Cin;
      a_ih0[i] = oh * p.stride - p.pad_t;
      a_iw0[i] = ow * p.stride - p.pad_l;
    } else {
      a_base[i] = p.A + (long long)m * p.lda;
      if (p.gate) a_gate[i] = p.gate + (long long)(m / p.rows_per_img) * p.K;
    }
  }
  int b_row[BL], b_kq[BL];
  bool b_ok[BL];
  const float* b_base[BL];
#pragma unroll
  for (int i = 0; i < BL; ++i) {
    int id = tid + i * 256;
    b_row[i] = id >> 2;
    b_kq[i] = (id & 3) * 4;
    int n = n0 + b_row[i];
    b_ok[i] = (n < p.N) && (!B_PARTIAL || id < BN * 4);
    b_base[i] = p.W + (long long)(b_ok[i] ? n : 0) * p.K;
  }

  // split-K: this CTA reduces k in [kbeg, kend) (the whole K without a split)
  const int kbeg = p.splitk > 1 ? blockIdx.z * p.k_chunk : 0;
  const int kend = p.splitk > 1 ? min(p.K, kbeg + p.k_chunk) : p.K;
  float4 a_reg[AL], b_reg[BL];
  auto load_slab = [&](int k0) {
#pragma unroll
    for (int i = 0; i < AL; ++i) {
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      int k = k0 + a_kq[i];
      if (a_ok[i] && k < kend) {
        if (p.conv) {
          int tap = k / p.Cin;
          int ci = k - tap * p.Cin;
          int kh = tap / p.KW, kw = tap - kh * p.KW;
          int ih = a_ih0[i] + kh, iw = a_iw0[i] + kw;
          if (ih >= 0 && ih < p.H && iw >= 0 && iw < p.Wd)
            v = __ldg(reinterpret_cast<const float4*>(a_base[i] + ((long long)ih * p.Wd + iw) * p.Cin + ci));
        } else {
          v = __ldg(reinterpret_cast<const float4*>(a_base[i] + k));
          if (a_gate[i]) {
            float4 g = __ldg(reinterpret_cast<const float4*>(a_gate[i] + k));
            v.x *= g.x; v.y *= g.y; v.z *= g.z; v.w *= g.w;
          }
        }
      }
      a_reg[i] = v;
    }
#pragma unroll
    for (int i = 0; i < BL; ++i) {
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      int k = k0 + b_kq[i];
      if (b_ok[i] && k < kend) v = __ldg(reinterpret_cast<const float4*>(b_base[i] + k));
      b_reg[i] = v;
    }
  };
  auto store_slab = [&]() {
#pragma unroll
    for (int i = 0; i < AL; ++i) {
      As[a_kq[i] + 0][a_row[i]] = a_reg[i].x;
      As[a_kq[i] + 1][a_row[i]] = a_reg[i].y;
      As[a_kq[i] + 2][a_row[i]] = a_reg[i].z;
      As[a_kq[i] + 3][a_row[i]] = a_reg[i].w;
    }
#pragma unroll
    for (int i = 0; i < BL; ++i) {
      if (!B_PARTIAL || tid + i * 256 < BN * 4) {
        Bs[b_kq[i] + 0][b_row[i]] = b_reg[i].x;
        Bs[b_kq[i] + 1][b_row[i]] = b_reg[i].y;
        Bs[b_kq[i] + 2][b_row[i]] = b_reg[i].z;
        Bs[b_kq[i] + 3][b_row[i]] = b_reg[i].w;
      }
    }
  };

  const int tx = tid % (BN / TN), ty = tid / (BN / TN);
  float acc[TM][TN];
#pragma unroll
  for (int i = 0; i < TM; ++i)
#pragma unroll
    for (int j = 0; j < TN; ++j) acc[i][j] = 0.f;

  load_slab(kbeg);
  store_slab();
  __syncthreads();
  for (int k0 = kbeg; k0 < kend; k0 += BK) {
    const bool more = k0 + BK < kend;
    if (more) load_slab(k0 + BK);
#pragma unroll
    for (int k = 0; k < BK; ++k) {
      float a[TM], b[TN];
#pragma unroll
      for (int i = 0; i < TM; i += 4) {
        float4 v = *reinterpret_cast<const float4*>(&As[k][ty * TM + i]);
        a[i] = v.x; a[i + 1] = v.y; a[i + 2] = v.z; a[i + 3] = v.w;
      }
#pragma unroll
      for (int j = 0; j < TN; j += 4) {
        float4 v = *reinterpret_cast<const float4*>(&Bs[k][tx * TN + j]);
        b[j] = v.x; b[j + 1] = v.y; b[j + 2] = v.z; b[j + 3] = v.w;
      }
#pragma unroll
      for (int i = 0; i < TM; ++i)
#pragma unroll
        for (int j = 0; j < TN; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
    }
    __syncthreads();
    if (more) {
      store_slab();
      __syncthreads();
    }
  }

  // ---- epilogue -----------------------------------------------------------
#pragma unroll
  for (int i = 0; i < TM; ++i) {
    int m = m0 + ty * TM + i;
    if (m >= p.M) continue;
#pragma unroll
    for (int j = 0; j < TN; ++j) {
      int n = n0 + tx * TN + j;
      if (n >= p.N) continue;
      float v = acc[i][j];
      if (p.splitk > 1) { p.ws[((long long)blockIdx.z * p.M + m) * p.N + n] = v; continue; }   // partial tile: epilogue in splitk_reduce
      if (p.scale) v = v * __ldg(p.scale + n) + __ldg(p.shift + n);
      else if (p.shift) v += __ldg(p.shift + n);
      v = act_apply(v, p.act);
      if (p.res) v += __ldg(p.res + (long long)m * p.ldr + n);
      p.C[(long long)m * p.ldc + n] = v;
    }
  }
}

// sums the split-K partials in split order and applies the GEMM epilogue
__global__ void __launch_bounds__(256) splitk_reduce_kernel(const GemmP p) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (long long)p.M * p.N) return;
  const int n = (int)(i % p.N);
  const long long m = i / p.N;
  float v = 0.f;
  for (int z = 0; z < p.splitk; ++z) v += p.ws[(long long)z * p.M * p.N + i];
  if (p.scale) v = v * __ldg(p.scale + n) + __ldg(p.shift + n);
  else if (p.shift) v += __ldg(p.shift + n);
  v = act_apply(v, p.act);
  if (p.res) v += __ldg(p.res + m * p.ldr + n);
  p.C[m * p.ldc + n] = v;
}

void launch_igemm_f32(const GemmP& p0, cudaStream_t st) {
  GemmP p = p0;
  p.splitk = 1; p.k_chunk = p.K;
  if (p.ws && p.K >= 256) {
    // tiles of the launch below; a launch of few tiles walks K serially in every CTA (the squeeze-excite FCs of a
    // 16-image batch are ONE tile over K = 1536): split K until ~240 CTAs exist
    const long long tiles = p.N <= 32 ? (long long)((p.M + 127) / 128) * ((p.N + 31) / 32)
                            : p.M >= 16384 ? (long long)((p.M + 127) / 128) * ((p.N + 63) / 64)
                                           : (long long)((p.M + 63) / 64) * ((p.N + 63) / 64);
    if (tiles < 120) {
      long long S = (240 + tiles - 1) / tiles;
      if (S > p.K / 64) S = p.K / 64;
      if (S > 32) S = 32;
      while (S > 1 && (long long)p.M * p.N * S > p.ws_floats) --S;
      if (S > 1) {
        p.k_chunk = (int)(((p.K + S - 1) / S + 15) / 16 * 16);
        p.splitk = (p.K + p.k_chunk - 1) / p.k_chunk;
        if (p.splitk <= 1) { p.splitk = 1; p.k_chunk = p.K; }
      }
    }
  }
  const unsigned gz = (unsigned)p.splitk;
  if (p.N <= 32) {
    dim3 g((p.M + 127) / 128, (p.N + 31) / 32, gz);
    igemm_f32_kernel<128, 32, 4, 4><<<g, 256, 0, st>>>(p);
  } else if (p.M >= 16384) {
    dim3 g((p.M + 127) / 128, (p.N + 63) / 64, gz);
    igemm_f32_kernel<128, 64, 8, 4><<<g, 256, 0, st>>>(p);
  } else {
    dim3 g((p.M + 63) / 64, (p.N + 63) / 64, gz);
    igemm_f32_kernel<64, 64, 4, 4><<<g, 256, 0, st>>>(p);
  }
  if (p.splitk > 1) {
    const long long n = (long long)p.M * p.N;
    splitk_reduce_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(p);
  }
}

// ===========================================================================
// 3. Depthwise 3x3 (+ folded BN / bias + activation), NHWC, float4 over channels
// ===========================================================================
__global__ void __launch_bounds__(256) dwconv3x3_f32_kernel(const DwP p) {
  const int C4 = p.C >> 2;
  long long total = (long long)p.B * p.OH * p.OW * C4;
  long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= total) return;
  int c = (int)(idx % C4) * 4;
  long long pix = idx / C4;
  int ow = (int)(pix % p.OW);
  int oh = (int)((pix / p.OW) % p.OH);
  int n = (int)(pix / ((long long)p.OW * p.OH));
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
  for (int kh = 0; kh < 3; ++kh) {
    int ih = oh * p.stride - p.pad_t + kh;
    if (ih < 0 || ih >= p.H) continue;
#pragma unroll
    for (int kw = 0; kw < 3; ++kw) {
      int iw = ow * p.stride - p.pad_l + kw;
      if (iw < 0 || iw >= p.Wd) continue;
      float4 x = __ldg(reinterpret_cast<const float4*>(p.in + (((long long)n * p.H + ih) * p.Wd + iw) * p.C + c));
      float4 w = __ldg(reinterpret_cast<const float4*>(p.w + (kh * 3 + kw) * p.C + c));
      acc.x = fmaf(x.x, w.x, acc.x); acc.y = fmaf(x.y, w.y, acc.y);
      acc.z = fmaf(x.z, w.z, acc.z); acc.w = fmaf(x.w, w.w, acc.w);
    }
  }
  float4 sc = __ldg(reinterpret_cast<const float4*>(p.scale + c));
  float4 sh = __ldg(reinterpret_cast<const float4*>(p.shift + c));
  float4 o;
  o.x = act_apply(acc.x * sc.x + sh.x, p.act);
  o.y = act_apply(acc.y * sc.y + sh.y, p.act);
  o.z = act_apply(acc.z * sc.z + sh.z, p.act);
  o.w = act_apply(acc.w * sc.w + sh.w, p.act);
  *reinterpret_cast<float4*>(p.out + (((long long)n * p.OH + oh) * p.OW + ow) * p.C + c) = o;
}

void launch_dwconv_f32(const DwP& p, cudaStream_t st) {
  long long total = (long long)p.B * p.OH * p.OW * (p.C / 4);
  dwconv3x3_f32_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(p);
}

// ===========================================================================
// 4. Squeeze-excite gate: sigmoid(W2 * silu(W1 * mean_hw(x) + b1) + b2)
//    one CTA per image; deterministic (no atomics).
// ===========================================================================
__global__ void __launch_bounds__(256) se_gate_f32_kernel(const float* __restrict__ x,  // [B,HW,C]
                                                          const float* __restrict__ w1,  // [R][C]
                                                          const float* __restrict__ b1,
                                                          const float* __restrict__ w2,  // [C][R]
                                                          const float* __restrict__ b2,
                                                          float* __restrict__ gate,      // [B][C]
                                                          int HW, int C, int R) {
  extern __shared__ float sm[];
  float* mean = sm;      // C
  float* red = sm + C;   // R
  const int n = blockIdx.x;
  const float* xp = x + (long long)n * HW * C;
  const float inv = 1.f / (float)HW;
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    float s = 0.f;
    for (int q = 0; q < HW; ++q) s += __ldg(xp + (long long)q * C + c);
    mean[c] = s * inv;
  }
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int r = warp; r < R; r += 8) {
    float s = 0.f;
    for (int c = lane; c < C; c += 32) s = fmaf(__ldg(w1 + (long long)r * C + c), mean[c], s);
    s = warp_sum(s);
    if (lane == 0) red[r] = act_apply(s + __ldg(b1 + r), ACT_SILU);
  }
  __syncthreads();
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    float s = __ldg(b2 + c);
    const float* wr = w2 + (long long)c * R;
    for (int r = 0; r < R; ++r) s = fmaf(__ldg(wr + r), red[r], s);
    gate[(long long)n * C + c] = 1.f / (1.f + expf(-s));
  }
}

void launch_se_gate_f32(const float* x, const float* w1, const float* b1, const float* w2,
                        const float* b2, float* gate, int B, int HW, int C, int R, cudaStream_t st) {
  se_gate_f32_kernel<<<B, 256, (C + R) * sizeof(float), st>>>(x, w1, b1, w2, b2, gate, HW, C, R);
}

// ===========================================================================
// 5. Max-pool 2x2 stride 2, NHWC (LiteSATRN ShallowCNN, LiteSATRN.py:29-59)
// ===========================================================================
__global__ void __launch_bounds__(256) maxpool2_f32_kernel(const float* __restrict__ in,
                                                           float* __restrict__ out, int B, int H, int W,
                                                           int C) {
  const int OH = H / 2, OW = W / 2, C4 = C / 4;
  long long total = (long long)B * OH * OW * C4;
  long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= total) return;
  int c = (int)(idx % C4) * 4;
  long long pix = idx / C4;
  int ow = (int)(pix % OW);
  int oh = (int)((pix / OW) % OH);
  int n = (int)(pix / ((long long)OW * OH));
  const float* base = in + (((long long)n * H + oh * 2) * W + ow * 2) * C + c;
  float4 a = __ldg(reinterpret_cast<const float4*>(base));
  float4 b = __ldg(reinterpret_cast<const float4*>(base + C));
  float4 d = __ldg(reinterpret_cast<const float4*>(base + (long long)W * C));
  float4 e = __ldg(reinterpret_cast<const float4*>(base + (long long)W * C + C));
  float4 o;
  o.x = fmaxf(fmaxf(a.x, b.x), fmaxf(d.x, e.x));
  o.y = fmaxf(fmaxf(a.y, b.y), fmaxf(d.y, e.y));
  o.z = fmaxf(fmaxf(a.z, b.z), fmaxf(d.z, e.z));
  o.w = fmaxf(fmaxf(a.w, b.w), fmaxf(d.w, e.w));
  *reinterpret_cast<float4*>(out + (((long long)n * OH + oh) * OW + ow) * C + c) = o;
}

void launch_maxpool2_f32(const float* in, float* out, int B, int H, int W, int C, cudaStream_t st) {
  long long total = (long long)B * (H / 2) * (W / 2) * (C / 4);
  maxpool2_f32_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(in, out, B, H, W, C);
}

// ===========================================================================
// 6. Adaptive 2-D positional encoding (:135-154): one CTA per image.
//    x NHWC [B, S=h*w, C]; gates = sigmoid(W1 relu(W0 mean + b0) + b1) [2C];
//    out = x + g[c]*PEh[row][c] + g[C+c]*PEw[col][c]
// ===========================================================================
__global__ void __launch_bounds__(1024) pe2d_f32_kernel(const float* __restrict__ x,
                                                       const float* __restrict__ w0,  // [C/2][C]
                                                       const float* __restrict__ b0,
                                                       const float* __restrict__ w1,  // [2C][C/2]
                                                       const float* __restrict__ b1,
                                                       const float* __restrict__ peh,  // [h][C]
                                                       const float* __restrict__ pew,  // [w][C]
                                                       float* __restrict__ out, int h, int w, int C) {
  extern __shared__ float sm[];
  float* mean = sm;            // C
  float* hid = sm + C;         // C/2
  float* g = hid + C / 2;      // 2C
  const int S = h * w, n = blockIdx.x;
  const float* xp = x + (long long)n * S * C;
  const float inv = 1.f / (float)S;
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    float s = 0.f;
    for (int q = 0; q < S; ++q) s += __ldg(xp + (long long)q * C + c);
    mean[c] = s * inv;
  }
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int nwarps = blockDim.x >> 5;
  for (int r = warp; r < C / 2; r += nwarps) {
    float s = 0.f;
    for (int c = lane; c < C; c += 32) s = fmaf(__ldg(w0 + (long long)r * C + c), mean[c], s);
    s = warp_sum(s);
    if (lane == 0) hid[r] = fmaxf(s + __ldg(b0 + r), 0.f);
  }
  __syncthreads();
  for (int r = warp; r < 2 * C; r += nwarps) {
    float s = 0.f;
    for (int c = lane; c < C / 2; c += 32) s = fmaf(__ldg(w1 + (long long)r * (C / 2) + c), hid[c], s);
    s = warp_sum(s);
    if (lane == 0) g[r] = 1.f / (1.f + expf(-(s + __ldg(b1 + r))));
  }
  __syncthreads();
  float* op = out + (long long)n * S * C;
  for (int i = threadIdx.x; i < S * C; i += blockDim.x) {
    int c = i % C, q = i / C;
    int row = q / w, col = q % w;
    float pos = g[c] * __ldg(peh + row * C + c) + g[C + c] * __ldg(pew + col * C + c);
    op[i] = pos + __ldg(xp + i);
  }
}

void launch_pe2d_f32(const float* x, const float* w0, const float* b0, const float* w1, const float* b1,
                     const float* peh, const float* pew, float* out, int B, int h, int w, int C,
                     cudaStream_t st) {
  int smem = (C + C / 2 + 2 * C) * sizeof(float);
  pe2d_f32_kernel<<<B, 1024, smem, st>>>(x, w0, b0, w1, b1, peh, pew, out, h, w, C);
}

// ===========================================================================
// 7. Row LayerNorm (eps 1e-5), optional residual, optional "scrambled" store
//    that realises the reference's raw reshape [B,HW,C] -> [B,C,H,W] (:269,
//    SURVEY F4) in NHWC terms: flat index f = q*C + ch of image b is written to
//    pixel p = f % S, channel c' = f / S.
// ===========================================================================
__device__ __forceinline__ void store_as(float* p, float v) { *p = v; }
__device__ __forceinline__ void store_as(eh_t* p, float v) { *p = eh_from_float(v); }

template <typename OutT>
__global__ void __launch_bounds__(256) layernorm_f32_generic_kernel(const float* __restrict__ x,
                                                            const float* __restrict__ res,
                                                            const float* __restrict__ gamma,
                                                            const float* __restrict__ beta,
                                                            OutT* __restrict__ out, int M, int C,
                                                            int scramble_S) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int m = blockIdx.x * 8 + warp;
  if (m >= M) return;
  const float* xp = x + (long long)m * C;
  const float* rp = res ? res + (long long)m * C : nullptr;
  float v[64];  // C <= 2048
  const int per = C / 32;
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < 64; ++i) {
    if (i < per) {
      float t = __ldg(xp + i * 32 + lane);
      if (rp) t += __ldg(rp + i * 32 + lane);
      v[i] = t;
      s += t;
    }
  }
  const float mean = warp_sum(s) / (float)C;
  float q = 0.f;
#pragma unroll
  for (int i = 0; i < 64; ++i)
    if (i < per) { float d = v[i] - mean; q = fmaf(d, d, q); }
  const float rstd = rsqrtf(warp_sum(q) / (float)C + 1e-5f);
#pragma unroll
  for (int i = 0; i < 64; ++i) {
    if (i < per) {
      int ch = i * 32 + lane;
      float o = (v[i] - mean) * rstd * __ldg(gamma + ch) + __ldg(beta + ch);
      if (scramble_S > 0) {
        int b = m / scramble_S, qd = m % scramble_S;
        long long f = (long long)qd * C + ch;
        int pp = (int)(f % scramble_S), cc = (int)(f / scramble_S);
        store_as(out + ((long long)b * scramble_S + pp) * C + cc, o);
      } else {
        store_as(out + (long long)m * C + ch, o);
      }
    }
  }
}

// PER = C / 32 values per lane (template: with a run-time bound the row lived in 64 registers per thread whatever C
// was -- 2 CTAs per SM -- and small-C rows, e.g. SwinTRN's 128-wide stage, paid 64 predicated iterations per pass).
// The accumulation order is the same for every PER, so results do not depend on the instantiation.
template <typename OutT, int PER>
__global__ void __launch_bounds__(256) layernorm_f32_kernel(const float* __restrict__ x,
                                                            const float* __restrict__ res,
                                                            const float* __restrict__ gamma,
                                                            const float* __restrict__ beta,
                                                            OutT* __restrict__ out, int M, int C,
                                                            int scramble_S) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int m = blockIdx.x * 8 + warp;
  if (m >= M) return;
  const float* xp = x + (long long)m * C;
  const float* rp = res ? res + (long long)m * C : nullptr;
  float v[PER];
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < PER; ++i) {
    float t = __ldg(xp + i * 32 + lane);
    if (rp) t += __ldg(rp + i * 32 + lane);
    v[i] = t;
    s += t;
  }
  const float mean = warp_sum(s) / (float)C;
  float q = 0.f;
#pragma unroll
  for (int i = 0; i < PER; ++i) { float d = v[i] - mean; q = fmaf(d, d, q); }
  const float rstd = rsqrtf(warp_sum(q) / (float)C + 1e-5f);
#pragma unroll
  for (int i = 0; i < PER; ++i) {
    int ch = i * 32 + lane;
    float o = (v[i] - mean) * rstd * __ldg(gamma + ch) + __ldg(beta + ch);
    if (scramble_S > 0) {
      int b = m / scramble_S, qd = m % scramble_S;
      long long f = (long long)qd * C + ch;
      int pp = (int)(f % scramble_S), cc = (int)(f / scramble_S);
      store_as(out + ((long long)b * scramble_S + pp) * C + cc, o);
    } else {
      store_as(out + (long long)m * C + ch, o);
    }
  }
}

template <typename OutT>
static void layernorm_launch(const float* x, const float* res, const float* gamma, const float* beta, OutT* out, int M, int C,
                             int scramble_S, cudaStream_t st) {
  const dim3 g((M + 7) / 8);
  const int per = C / 32;  // C is a multiple of 32, at most 2048
  if (per <= 4 && per * 32 == C) {
    if (per == 4) layernorm_f32_kernel<OutT, 4><<<g, 256, 0, st>>>(x, res, gamma, beta, out, M, C, scramble_S);
    else if (per == 2) layernorm_f32_kernel<OutT, 2><<<g, 256, 0, st>>>(x, res, gamma, beta, out, M, C, scramble_S);
    else if (per == 1) layernorm_f32_kernel<OutT, 1><<<g, 256, 0, st>>>(x, res, gamma, beta, out, M, C, scramble_S);
    else layernorm_f32_kernel<OutT, 3><<<g, 256, 0, st>>>(x, res, gamma, beta, out, M, C, scramble_S);
  } else if (per == 8) layernorm_f32_kernel<OutT, 8><<<g, 256, 0, st>>>(x, res, gamma, beta, out, M, C, scramble_S);
  else if (per == 16) layernorm_f32_kernel<OutT, 16><<<g, 256, 0, st>>>(x, res, gamma, beta, out, M, C, scramble_S);
  else if (per == 32) layernorm_f32_kernel<OutT, 32><<<g, 256, 0, st>>>(x, res, gamma, beta, out, M, C, scramble_S);
  else if (per == 64) layernorm_f32_kernel<OutT, 64><<<g, 256, 0, st>>>(x, res, gamma, beta, out, M, C, scramble_S);
  else layernorm_f32_generic_kernel<OutT><<<g, 256, 0, st>>>(x, res, gamma, beta, out, M, C, scramble_S);
}

void launch_layernorm_f32(const float* x, const float* res, const float* gamma, const float* beta,
                          float* out, int M, int C, int scramble_S, cudaStream_t st) {
  layernorm_launch<float>(x, res, gamma, beta, out, M, C, scramble_S, st);
}

// Scrambled store (the reference's raw reshape, SURVEY F4) for the bf16 path: one CTA per image normalises its S
// rows into shared memory laid out as the flat index f = token * C + ch seen as [f / S][f % S], then writes
// out[(f % S) * C + f / S] with consecutive lanes on consecutive addresses -- a tiled transpose instead of
// S * C scattered 2-byte stores.
__global__ void __launch_bounds__(256) layernorm_scramble_bf16_kernel(const float* __restrict__ x, const float* __restrict__ res,
                                                                      const float* __restrict__ gamma,
                                                                      const float* __restrict__ beta,
                                                                      eh_t* __restrict__ out, int S, int C) {
  extern __shared__ eh_t ln_tile[];  // [C][S + 2]
  const int b = blockIdx.x, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int per = C / 32, LD = S + 2;
  for (int qd = warp; qd < S; qd += 8) {
    const float* xp = x + ((long long)b * S + qd) * C;
    const float* rp = res ? res + ((long long)b * S + qd) * C : nullptr;
    float v[16];  // C <= 512
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < 16; ++i)
      if (i < per) {
        float t = __ldg(xp + i * 32 + lane);
        if (rp) t += __ldg(rp + i * 32 + lane);
        v[i] = t;
        s += t;
      }
    const float mean = warp_sum(s) / (float)C;
    float q = 0.f;
#pragma unroll
    for (int i = 0; i < 16; ++i)
      if (i < per) { float d = v[i] - mean; q = fmaf(d, d, q); }
    const float rstd = rsqrtf(warp_sum(q) / (float)C + 1e-5f);
#pragma unroll
    for (int i = 0; i < 16; ++i)
      if (i < per) {
        const int ch = i * 32 + lane;
        const int f = qd * C + ch;
        ln_tile[(f / S) * LD + f % S] = eh_from_float((v[i] - mean) * rstd * __ldg(gamma + ch) + __ldg(beta + ch));
      }
  }
  __syncthreads();
  eh_t* op = out + (long long)b * S * C;
  for (int g = threadIdx.x; g < S * C; g += 256) {  // g = pp * C + cc
    const int pp = g / C, cc = g - pp * C;
    op[g] = ln_tile[cc * LD + pp];
  }
}

void launch_layernorm_bf16out(const float* x, const float* res, const float* gamma, const float* beta,
                              eh_t* out, int M, int C, int scramble_S, cudaStream_t st) {
  const size_t scr_smem = (size_t)C * (scramble_S + 2) * 2;
  static SmemOptIn scr_opt;
  if (scramble_S > 0 && C <= 512 && C % 32 == 0 && M % scramble_S == 0 && scr_smem <= 160 * 1024 &&
      scr_opt.ensure(layernorm_scramble_bf16_kernel, scr_smem) == cudaSuccess) {
    layernorm_scramble_bf16_kernel<<<M / scramble_S, 256, scr_smem, st>>>(x, res, gamma, beta, out,
                                                                                               scramble_S, C);
    return;
  }
  layernorm_launch<eh_t>(x, res, gamma, beta, out, M, C, scramble_S, st);
}

// ===========================================================================
// 8. Encoder self-attention (:164-172,:198-228): one CTA per (image, head);
//    S tokens x HD=64; scores divided by sqrt(heads*HD).
// ===========================================================================
// DROP (training step only): attention dropout on the probabilities [B, heads, S, S] -- the softmax sum is taken over the
// undropped probabilities, P.M.scale multiplies V.
template <typename OutT, bool DROP = false>
__global__ void __launch_bounds__(128) enc_attn_f32_kernel(const float* __restrict__ qkv,  // [B*S, 3*D]
                                                           OutT* __restrict__ out,        // [B*S, D]
                                                           int S, int D, int heads, float temperature, DropP drop) {
  extern __shared__ float sm[];
  const int HD = D / heads;  // 64
  const int LDS_ = HD + 1;
  float* Q = sm;
  float* K = Q + S * LDS_;
  float* V = K + S * LDS_;
  float* P = V + S * LDS_;  // [4 warps][S]
  const int b = blockIdx.x / heads, hh = blockIdx.x % heads;
  const float* base = qkv + (long long)b * S * 3 * D + hh * HD;
  for (int i = threadIdx.x; i < S * HD; i += blockDim.x) {
    int r = i / HD, c = i % HD;
    const float* rp = base + (long long)r * 3 * D + c;
    Q[r * LDS_ + c] = __ldg(rp);
    K[r * LDS_ + c] = __ldg(rp + D);
    V[r * LDS_ + c] = __ldg(rp + 2 * D);
  }
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float* Pw = P + warp * S;
  for (int i = warp; i < S; i += 4) {
    float mx = -INFINITY;
    for (int j = lane; j < S; j += 32) {
      float s = 0.f;
      for (int c = 0; c < HD; ++c) s = fmaf(Q[i * LDS_ + c], K[j * LDS_ + c], s);
      s = s / temperature;
      Pw[j] = s;
      mx = fmaxf(mx, s);
    }
    mx = warp_max(mx);
    float sum = 0.f;
    for (int j = lane; j < S; j += 32) {
      float e = expf(Pw[j] - mx);
      Pw[j] = e;
      sum += e;
    }
    sum = warp_sum(sum);
    if constexpr (DROP) {
      for (int j = lane; j < S; j += 32) Pw[j] *= drop_factor(drop, ((long long)blockIdx.x * S + i) * S + j) != 0.f ? 1.f : 0.f;
    }
    __syncwarp();
    for (int c = lane; c < HD; c += 32) {
      float acc = 0.f;
      for (int j = 0; j < S; ++j) {
        if constexpr (DROP) acc = fmaf(__fmul_rn(Pw[j] / sum, drop.scale), V[j * LDS_ + c], acc);
        else acc = fmaf(Pw[j] / sum, V[j * LDS_ + c], acc);
      }
      store_as(out + ((long long)b * S + i) * D + hh * HD + c, acc);
    }
    __syncwarp();
  }
}

template <typename OutT>
static void enc_attn_launch(const float* qkv, OutT* out, int B, int S, int D, int heads, cudaStream_t st) {
  int HD = D / heads;
  size_t smem = (size_t)(3 * S * (HD + 1) + 4 * S) * sizeof(float);
  static SmemOptIn opt;
  opt.ensure(enc_attn_f32_kernel<OutT>, smem);
  enc_attn_f32_kernel<OutT><<<B * heads, 128, smem, st>>>(qkv, out, S, D, heads, sqrtf((float)D), DropP{});
}
void launch_enc_attn_f32(const float* qkv, float* out, int B, int S, int D, int heads, cudaStream_t st) {
  enc_attn_launch<float>(qkv, out, B, S, D, heads, st);
}
void launch_enc_attn_f32_drop(const float* qkv, float* out, int B, int S, int D, int heads, const DropP& drop, cudaStream_t st) {
  const size_t smem = (size_t)(3 * S * (D / heads + 1) + 4 * S) * sizeof(float);
  static SmemOptIn opt;
  opt.ensure(enc_attn_f32_kernel<float, true>, smem);
  enc_attn_f32_kernel<float, true><<<B * heads, 128, smem, st>>>(qkv, out, S, D, heads, sqrtf((float)D), drop);
}
void launch_enc_attn_bf16out(const float* qkv, eh_t* out, int B, int S, int D, int heads, cudaStream_t st) {
  enc_attn_launch<eh_t>(qkv, out, B, S, D, heads, st);
}

// ===========================================================================
// 9. Decoder: small-M GEMM with optional LayerNorm-on-load, bias, ReLU,
//    residual and segmented output (KV-cache scatter).  Tile 32 x 32, the 8
//    warps split K; lane = output column.
// ===========================================================================
constexpr int DG_BM = 32, DG_BN = 32, DG_KC = 512;  // K chunk = widest LayerNorm row (SwinTRN decoder: 512)

__global__ void __launch_bounds__(256) dec_gemm_f32_kernel(const DecGemmP p) {
  extern __shared__ __align__(16) float smem_raw[];  // DG_BM * (DG_KC + 4) floats
  float (*As)[DG_KC + 4] = reinterpret_cast<float (*)[DG_KC + 4]>(smem_raw);
  float (*red)[DG_BM][DG_BN] = reinterpret_cast<float (*)[DG_BM][DG_BN]>(smem_raw);  // reused after the K loop
  static_assert(8 * DG_BM * DG_BN <= DG_BM * (DG_KC + 4), "partials must fit in the A buffer");
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int m0 = blockIdx.x * DG_BM, n0 = blockIdx.y * DG_BN;
  const int n = n0 + lane;
  const bool n_ok = n < p.N;
  float acc[DG_BM];
#pragma unroll
  for (int r = 0; r < DG_BM; ++r) acc[r] = 0.f;

  for (int kc = 0; kc < p.K; kc += DG_KC) {
    const int kn = min(DG_KC, p.K - kc);  // multiple of 32
    // ---- stage A chunk (row-major) -----------------------------------------
    for (int i = tid; i < DG_BM * (DG_KC / 4); i += 256) {
      int r = i / (DG_KC / 4), k4 = (i % (DG_KC / 4)) * 4;
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (m0 + r < p.M && k4 < kn) v = __ldg(reinterpret_cast<const float4*>(p.A + (long long)(m0 + r) * p.lda + kc + k4));
      *reinterpret_cast<float4*>(&As[r][k4]) = v;
    }
    __syncthreads();
    if (p.ln_g) {  // LayerNorm over the full row (K == row width <= DG_KC)
      for (int r = warp; r < DG_BM; r += 8) {
        float s = 0.f;
        for (int k = lane; k < kn; k += 32) s += As[r][k];
        float mean = warp_sum(s) / (float)kn;
        float q = 0.f;
        for (int k = lane; k < kn; k += 32) { float d = As[r][k] - mean; q = fmaf(d, d, q); }
        float rstd = rsqrtf(warp_sum(q) / (float)kn + 1e-5f);
        for (int k = lane; k < kn; k += 32) {
          float o = (As[r][k] - mean) * rstd * __ldg(p.ln_g + k) + __ldg(p.ln_b + k);
          As[r][k] = o;
          if (p.a_norm_out && blockIdx.y == 0 && m0 + r < p.M) p.a_norm_out[(long long)(m0 + r) * kn + k] = o;
        }
      }
      __syncthreads();
    }
    // ---- each warp owns a K slice of the chunk -----------------------------
    const int ks = kn / 8;  // multiple of 4
    const int kb = warp * ks;
    if (n_ok) {
      // the weight rows of the NEXT two k-groups are requested before the current group's FMAs: the loop is a chain of
      // L2 round trips otherwise (16 per warp at K = 512).  Accumulation order is unchanged.
      const float* wbase = p.Wt + (long long)kc * p.N + n;
      auto ldw = [&](int k, float (&w)[4]) {
        if (k < kb + ks) {
          const float* wp = wbase + (long long)k * p.N;
          w[0] = __ldg(wp); w[1] = __ldg(wp + p.N); w[2] = __ldg(wp + 2LL * p.N); w[3] = __ldg(wp + 3LL * p.N);
        }
      };
      float wa[4] = {0.f, 0.f, 0.f, 0.f}, wb[4] = {0.f, 0.f, 0.f, 0.f}, wc[4] = {0.f, 0.f, 0.f, 0.f};
      ldw(kb, wa);
      ldw(kb + 4, wb);
      for (int k = kb; k < kb + ks; k += 4) {
        ldw(k + 8, wc);
#pragma unroll
        for (int r = 0; r < DG_BM; ++r) {
          float4 a = *reinterpret_cast<const float4*>(&As[r][k]);
          acc[r] = fmaf(a.x, wa[0], acc[r]);
          acc[r] = fmaf(a.y, wa[1], acc[r]);
          acc[r] = fmaf(a.z, wa[2], acc[r]);
          acc[r] = fmaf(a.w, wa[3], acc[r]);
        }
#pragma unroll
        for (int i = 0; i < 4; ++i) { wa[i] = wb[i]; wb[i] = wc[i]; }
      }
    }
    __syncthreads();
  }
#pragma unroll
  for (int r = 0; r < DG_BM; ++r) red[warp][r][lane] = acc[r];
  __syncthreads();
  // ---- combine the 8 K-slices in a fixed order + epilogue -------------------
  for (int i = tid; i < DG_BM * DG_BN; i += 256) {
    int r = i / DG_BN, c = i % DG_BN;
    int m = m0 + r, nn = n0 + c;
    if (m >= p.M || nn >= p.N) continue;
    float v = red[0][r][c];
#pragma unroll
    for (int wv = 1; wv < 8; ++wv) v += red[wv][r][c];
    if (p.bias) v += __ldg(p.bias + nn);
    v = act_apply(v, p.act);
    if (p.res) v += __ldg(p.res + (long long)m * p.ldr + nn);
#pragma unroll
    for (int s = 0; s < 4; ++s) {
      if (s < p.nseg && nn >= p.seg[s].n_begin && nn < p.seg[s].n_end) {
        long long off = (long long)m * p.seg[s].row_stride + (nn - p.seg[s].n_begin);
        if (p.row_slot) off += (long long)__ldg(p.row_slot + m) * p.seg[s].slot_stride;
        p.seg[s].dst[off] = v;
      }
    }
  }
}

void launch_dec_gemm_f32(const DecGemmP& p, cudaStream_t st) {
  dim3 g((p.M + DG_BM - 1) / DG_BM, (p.N + DG_BN - 1) / DG_BN);
  static SmemOptIn opt;
  const int smem = DG_BM * (DG_KC + 4) * (int)sizeof(float);
  opt.ensure(dec_gemm_f32_kernel, (size_t)smem, true);
  dec_gemm_f32_kernel<<<g, 256, smem, st>>>(p);
}

// ===========================================================================
// 10. Decoder attention over a row cache (+ optional extra "current" key):
//     one warp per (query row, head), HD = 32 -> lane = channel for P.V.
//     Implements :164-172 on the recurrence of SURVEY App. A.4.
// ===========================================================================
// DROP (training step only): attention dropout on the probabilities, logical layout [images, heads, q_per_img,
// rows_per_img] (teacher forcing: [B, H, L, L] / [B, H, L, S]); the softmax sum is over the undropped probabilities.
template <int HD, bool DROP = false>
__global__ void __launch_bounds__(256) dec_attn_f32_kernel(const AttnP p, DropP drop) {
  extern __shared__ float sm[];  // [8 warps][max_keys]
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int gw = blockIdx.x * 8 + warp;
  const int m = gw / p.heads, hh = gw % p.heads;
  if (m >= p.M) return;
  const int img = m / p.q_per_img;
  const int nh = p.causal_L > 0 ? (m % p.causal_L) + 1 : (p.hist_len ? __ldg(p.hist_len + m) : p.n_hist);
  const unsigned char* kmask = p.key_mask ? p.key_mask + (long long)img * p.rows_per_img : nullptr;
  const int nk = nh + (p.cur_k ? 1 : 0);
  float* sc = sm + (size_t)warp * (p.rows_per_img + 1);
  constexpr int PER = HD / 32;
  // q in registers (every lane holds the whole head vector)
  float qv[HD];
  {
    const float* qp = p.q + (long long)m * p.ldq + hh * HD;
#pragma unroll
    for (int c = 0; c < HD; c += 4) {
      float4 t = __ldg(reinterpret_cast<const float4*>(qp + c));
      qv[c] = t.x; qv[c + 1] = t.y; qv[c + 2] = t.z; qv[c + 3] = t.w;
    }
  }
  const float* kbase = p.kcache + (long long)img * p.rows_per_img * p.D + hh * HD;
  const float* vbase = p.vcache + (long long)img * p.rows_per_img * p.D + hh * HD;
  const int* chain = p.chain ? p.chain + (long long)m * p.chain_stride : nullptr;
  float mx = -INFINITY;
  for (int j = lane; j < nk; j += 32) {
    const float* kp;
    if (j < nh) kp = kbase + (long long)(chain ? __ldg(chain + j) : j) * p.D;
    else kp = p.cur_k + (long long)m * p.ld_cur + hh * HD;
    float s = 0.f;
#pragma unroll
    for (int c = 0; c < HD; c += 4) {
      float4 t = __ldg(reinterpret_cast<const float4*>(kp + c));
      s = fmaf(qv[c], t.x, s); s = fmaf(qv[c + 1], t.y, s);
      s = fmaf(qv[c + 2], t.z, s); s = fmaf(qv[c + 3], t.w, s);
    }
    s = s / p.temperature;
    if (kmask && j < nh && kmask[j]) s = -INFINITY;  // masked_fill(-inf) (:168)
    sc[j] = s;
    mx = fmaxf(mx, s);
  }
  mx = warp_max(mx);
  float sum = 0.f;
  for (int j = lane; j < nk; j += 32) {
    float e = expf(sc[j] - mx);
    sc[j] = e;
    sum += e;
  }
  sum = warp_sum(sum);
  if constexpr (DROP) {
    const long long row = ((long long)img * p.heads + hh) * p.q_per_img + m % p.q_per_img;
    for (int j = lane; j < nk; j += 32) sc[j] *= drop_factor(drop, row * p.rows_per_img + j) != 0.f ? 1.f : 0.f;
  }
  __syncwarp();
  float acc[PER];
#pragma unroll
  for (int i = 0; i < PER; ++i) acc[i] = 0.f;
  for (int j = 0; j < nk; ++j) {
    const float* vp;
    if (j < nh) vp = vbase + (long long)(chain ? __ldg(chain + j) : j) * p.D;
    else vp = p.cur_v + (long long)m * p.ld_cur + hh * HD;
    float pj = sc[j] / sum;
    if constexpr (DROP) pj = __fmul_rn(pj, drop.scale);
#pragma unroll
    for (int i = 0; i < PER; ++i) acc[i] = fmaf(pj, __ldg(vp + i * 32 + lane), acc[i]);
  }
#pragma unroll
  for (int i = 0; i < PER; ++i) p.out[(long long)m * p.ldo + hh * HD + i * 32 + lane] = acc[i];
}

void launch_dec_attn_f32(const AttnP& p, int head_dim, cudaStream_t st) {
  int warps = p.M * p.heads;
  size_t smem = (size_t)8 * (p.rows_per_img + 1) * sizeof(float);
  if (head_dim == 32) dec_attn_f32_kernel<32><<<(warps + 7) / 8, 256, smem, st>>>(p, DropP{});
  else dec_attn_f32_kernel<64><<<(warps + 7) / 8, 256, smem, st>>>(p, DropP{});
}
void launch_dec_attn_f32_drop(const AttnP& p, int head_dim, const DropP& drop, cudaStream_t st) {
  const int warps = p.M * p.heads;
  const size_t smem = (size_t)8 * (p.rows_per_img + 1) * sizeof(float);
  if (head_dim == 32) dec_attn_f32_kernel<32, true><<<(warps + 7) / 8, 256, smem, st>>>(p, drop);
  else dec_attn_f32_kernel<64, true><<<(warps + 7) / 8, 256, smem, st>>>(p, drop);
}

// ===========================================================================
// 11. Token embedding * sqrt(D) + 1-D positional row (:480-483, :420-426)
// ===========================================================================
__global__ void __launch_bounds__(256) dec_embed_f32_kernel(const int* __restrict__ tok,  // [M] or null
                                                            const long long* __restrict__ tok64,
                                                            int fixed_token, const float* __restrict__ emb,
                                                            const float* __restrict__ pe,  // [len][D]
                                                            int pos, const int* __restrict__ pos_arr,
                                                            int pos_mod, float scale, float* __restrict__ x,
                                                            int M, int D) {
  int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= M * D) return;
  int m = idx / D, d = idx % D;
  int t = tok ? __ldg(tok + m) : (tok64 ? (int)tok64[m] : fixed_token);
  int ps = pos_arr ? __ldg(pos_arr + m) : (pos_mod > 0 ? m % pos_mod : pos);
  x[idx] = __ldg(emb + (long long)t * D + d) * scale + __ldg(pe + (long long)ps * D + d);
}

void launch_dec_embed_f32(const int* tok, const long long* tok64, int fixed_token, const float* emb,
                          const float* pe, int pos, const int* pos_arr, int pos_mod, float scale, float* x,
                          int M, int D, cudaStream_t st) {
  dec_embed_f32_kernel<<<(M * D + 255) / 256, 256, 0, st>>>(tok, tok64, fixed_token, emb, pe, pos, pos_arr,
                                                            pos_mod, scale, x, M, D);
}

// ===========================================================================
// 12. Greedy pick (:556-557 / decoding.py:38-40): first index of the row
//     maximum; writes the int64 token output, the next input token (argmax or
//     forced) and the next step's embedded input.
// ===========================================================================
__global__ void __launch_bounds__(256) dec_argmax_embed_kernel(const float* __restrict__ logits,
                                                               long long ld_logits, int V,
                                                               long long* __restrict__ tokens_out,
                                                               long long ld_tok, const long long* __restrict__ forced,
                                                               long long ld_forced, int* __restrict__ cur_tok,
                                                               const float* __restrict__ emb,
                                                               const float* __restrict__ pe_next, float scale,
                                                               float* __restrict__ x, int M, int D) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int m = blockIdx.x * 8 + warp;
  if (m >= M) return;
  const float* lp = logits + (long long)m * ld_logits;
  float best = -INFINITY;
  int bi = 0x7fffffff;
  for (int i = lane; i < V; i += 32) {
    float v = lp[i];
    if (v > best) { best = v; bi = i; }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    float ob = __shfl_xor_sync(0xffffffffu, best, o);
    int oi = __shfl_xor_sync(0xffffffffu, bi, o);
    if (ob > best || (ob == best && oi < bi)) { best = ob; bi = oi; }
  }
  if (bi < 0 || bi >= V) bi = 0;  // all-NaN row: keep the lookup in range
  int nxt = bi;
  if (forced) nxt = (int)forced[(long long)m * ld_forced];
  if (lane == 0) {
    if (tokens_out) tokens_out[(long long)m * ld_tok] = bi;
    cur_tok[m] = nxt;
  }
  if (pe_next) {
    for (int d = lane; d < D; d += 32)
      x[(long long)m * D + d] = __ldg(emb + (long long)nxt * D + d) * scale + __ldg(pe_next + d);
  }
}

void launch_dec_argmax_embed(const float* logits, long long ld_logits, int V, long long* tokens_out,
                             long long ld_tok, const long long* forced, long long ld_forced, int* cur_tok,
                             const float* emb, const float* pe_next, float scale, float* x, int M, int D,
                             cudaStream_t st) {
  dec_argmax_embed_kernel<<<(M + 7) / 8, 256, 0, st>>>(logits, ld_logits, V, tokens_out, ld_tok, forced,
                                                       ld_forced, cur_tok, emb, pe_next, scale, x, M, D);
}


// pad_mask (:469-473): key j of a text row is masked when text[j] == PAD and j > 0
__global__ void __launch_bounds__(256) pad_mask_kernel(const long long* __restrict__ text, unsigned char* __restrict__ mask,
                                                       int B, int L, int pad_id) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B * L) return;
  mask[i] = (text[i] == pad_id && (i % L) != 0) ? 1 : 0;
}
void launch_pad_mask(const long long* text, unsigned char* mask, int B, int L, int pad_id, cudaStream_t st) {
  pad_mask_kernel<<<(B * L + 255) / 256, 256, 0, st>>>(text, mask, B, L, pad_id);
}

// Stop-at-<EOS> contract on a greedy result (one block per image): len = index of the first `eos` in stop[b] + 1, or
// steps; tokens after it become `pad`, logits rows after it 0.  have_len: lengths[b] is given (the stop-at-<EOS> kernel
// wrote only the rows up to it), else it is found in stop[] (the tokens, or the forced sequence) and written.
__global__ void __launch_bounds__(256) eos_finalize_kernel(float* __restrict__ logits, long long* __restrict__ tokens,
                                                           int* __restrict__ lengths, const long long* __restrict__ stop,
                                                           int steps, int V, int eos, int pad, int have_len) {
  __shared__ int first;
  const int b = blockIdx.x;
  if (threadIdx.x == 0) first = steps;
  __syncthreads();
  if (!have_len) {
    for (int t = threadIdx.x; t < steps; t += blockDim.x)
      if (stop[(size_t)b * steps + t] == eos) atomicMin(&first, t + 1);
    __syncthreads();
    if (threadIdx.x == 0) lengths[b] = first;
  }
  const int len = have_len ? lengths[b] : first;
  for (int t = len + threadIdx.x; t < steps; t += blockDim.x) tokens[(size_t)b * steps + t] = pad;
  if (logits) {
    float* row = logits + (size_t)b * steps * V;
    for (size_t i = (size_t)len * V + threadIdx.x; i < (size_t)steps * V; i += blockDim.x) row[i] = 0.f;
  }
}
void launch_eos_finalize(float* logits, long long* tokens, int* lengths, const long long* stop, int B, int steps, int V,
                         int eos, int pad, bool have_len, cudaStream_t st) {
  eos_finalize_kernel<<<B, 256, 0, st>>>(logits, tokens, lengths, stop, steps, V, eos, pad, have_len ? 1 : 0);
}

// ===========================================================================
// DecodingManager.sift + MemoryNode.record/_look_back (postprocessing/postprocessing.py:193-233,
// :303-391) fused with the next step's embedding: one warp per row.  In place: the row of logits becomes the
// row of masked softmax probabilities (what the reference's forward returns when a manager is attached,
// EfficientSATRN.py:553-555); the constrained argmax (first maximum, like torch.argmax) is the next input token.
// state[m] = {current token, run length, #'{', #'}'} (MemoryNode.__init__: <SOS>, 1, 0, 0).
// ===========================================================================
__global__ void __launch_bounds__(256) dec_sift_embed_kernel(float* __restrict__ logits, long long ld_logits, int V,
                                                             long long* __restrict__ tokens_out, long long ld_tok,
                                                             int4* __restrict__ state, const int* __restrict__ flags,
                                                             const int* __restrict__ limit, SiftIds ids,
                                                             int* __restrict__ cur_tok, const float* __restrict__ emb,
                                                             const float* __restrict__ pe_next, float scale,
                                                             float* __restrict__ x, int M, int D) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int m = blockIdx.x * 8 + warp;
  if (m >= M) return;
  float* lp = logits + (long long)m * ld_logits;
  int4 stt = state[m];  // x = current token, y = run length, z = '{' count, w = '}' count
  const int cur = stt.x;
  const int cf = (cur >= 0 && cur < V) ? __ldg(flags + cur) : 0;
  const int clim = (cur >= 0 && cur < V) ? __ldg(limit + cur) : 0;
  // softmax (F.softmax, :216)
  float mx = -INFINITY;
  for (int i = lane; i < V; i += 32) mx = fmaxf(mx, lp[i]);
  mx = warp_max(mx);
  float sum = 0.f;
  for (int i = lane; i < V; i += 32) sum += expf(lp[i] - mx);
  sum = warp_sum(sum);
  float best = -INFINITY;
  int bi = 0x7fffffff;
  for (int i = lane; i < V; i += 32) {
    // MemoryNode._look_back (:327-391)
    bool black = (i == ids.sos) || (i == ids.empty) || (i == ids.rbrace && stt.z == stt.w);
    if (cur == ids.eos) {
    } else if (cur == ids.sos) {
      black = black || (__ldg(flags + i) & 1);
    } else if (cf & 2) {
      black = black || (i != ids.underbar);
    } else if (cf & 4) {
      black = black || (i != ids.lbrace);
    } else {
      if ((cf & 8) && i == ids.underbar) black = true;
      if ((cf & 16) && i == ids.lbrace) black = true;
      if (clim > 0 && stt.y >= clim && i == cur) black = true;
    }
    const float pv = black ? 0.f : expf(lp[i] - mx) / sum;
    lp[i] = pv;
    if (pv > best) { best = pv; bi = i; }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    float ob = __shfl_xor_sync(0xffffffffu, best, o);
    int oi = __shfl_xor_sync(0xffffffffu, bi, o);
    if (ob > best || (ob == best && oi < bi)) { best = ob; bi = oi; }
  }
  if (bi < 0 || bi >= V) bi = 0;
  if (lane == 0) {  // MemoryNode.record (:303-325)
    stt.y = (bi == cur) ? stt.y + 1 : 1;
    if (bi == ids.lbrace) stt.z += 1;
    else if (bi == ids.rbrace) stt.w += 1;
    stt.x = bi;
    state[m] = stt;
    if (tokens_out) tokens_out[(long long)m * ld_tok] = bi;
    cur_tok[m] = bi;
  }
  if (pe_next) {
    for (int d = lane; d < D; d += 32)
      x[(long long)m * D + d] = __ldg(emb + (long long)bi * D + d) * scale + __ldg(pe_next + d);
  }
}

void launch_dec_sift_embed(float* logits, long long ld_logits, int V, long long* tokens_out, long long ld_tok, int4* state,
                           const int* flags, const int* limit, const SiftIds& ids, int* cur_tok, const float* emb,
                           const float* pe_next, float scale, float* x, int M, int D, cudaStream_t st) {
  dec_sift_embed_kernel<<<(M + 7) / 8, 256, 0, st>>>(logits, ld_logits, V, tokens_out, ld_tok, state, flags, limit, ids,
                                                     cur_tok, emb, pe_next, scale, x, M, D);
}

__global__ void sift_state_init_kernel(int4* state, int M, int sos) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < M) state[i] = make_int4(sos, 1, 0, 0);
}
void launch_sift_state_init(int4* state, int M, int sos, cudaStream_t st) {
  sift_state_init_kernel<<<(M + 255) / 256, 256, 0, st>>>(state, M, sos);
}

}  // namespace frx
