// common.cuh -- shared declarations for the frx CUDA library (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <stdint.h>

#if defined(__CUDA_ARCH__) && (__CUDA_ARCH__ < 1000)
#error "frx is written for sm_100a (B200) only"
#endif

namespace frx {

enum Act : int { ACT_NONE = 0, ACT_RELU = 1, ACT_SILU = 2, ACT_SIGMOID = 3, ACT_GELU = 4 };

__device__ __forceinline__ float act_apply(float v, int act) {
  switch (act) {
    case ACT_RELU: return fmaxf(v, 0.f);
    case ACT_SILU: return v / (1.f + expf(-v));
    case ACT_SIGMOID: return 1.f / (1.f + expf(-v));
    case ACT_GELU: return 0.5f * v * (1.f + erff(v * 0.70710678118654752440f));  // exact GELU (SWIN.py:30)
    default: return v;
  }
}

// cudaFuncSetAttribute(MaxDynamicSharedMemorySize) is a PER-DEVICE setting: remember what each call site has opted
// into per device, so a handle on a second GPU of the same process (model.to("cuda:1")) configures its own copy.
struct SmemOptIn {
  size_t bytes[64] = {};
  template <class Kernel>
  cudaError_t ensure(Kernel kernel, size_t smem, bool always = false) {
    int dev = 0;
    cudaGetDevice(&dev);
    dev &= 63;
    if ((!always && smem <= 48 * 1024) || (bytes[dev] != 0 && smem <= bytes[dev])) return cudaSuccess;
    cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e == cudaSuccess) bytes[dev] = smem;
    return e;
  }
};

// ---------------------------------------------------------------------------
// 16-bit storage / tensor-core operand type of the ENCODER side of the 16-bit mode (conv trunk, encoder layers, the
// teacher-forced decoder's GEMMs, SwinTRN / LiteSATRN encoders): IEEE fp16 by default.  bf16 and fp16 run at the same
// tensor-core rate (tcgen05 kind::f16, mma.sync m16n8k16) and occupy the same bytes, but fp16 keeps 11 significand bits
// against bf16's 8: on the synthetic checkpoint the encoder memory lands within 1.1 % (rel-L2) of the fp32 reference
// instead of 8-9 % (tools/bf16_yardstick.py: 0.080 is the floor of ANY bf16-operand pipeline).  BatchNorm-folded
// activations are O(1..100), far inside fp16's range; conversions saturate (cvt.rn.satfinite) instead of producing inf.
// The persistent decode kernel (KV cache, fragment-packed weights) stays bf16.  -DFRX_ENC_FP16=0 restores a bf16 encoder.
// ---------------------------------------------------------------------------
#ifndef FRX_ENC_FP16
#define FRX_ENC_FP16 1
#endif
#if FRX_ENC_FP16
typedef __half eh_t;
typedef __half2 eh2_t;
#define FRX_EH_PTX "f16"
__device__ __forceinline__ uint32_t eh2_pack(float lo, float hi) {
  uint32_t r;
  asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;\n" : "=r"(r) : "f"(hi), "f"(lo));
  return r;
}
__device__ __forceinline__ eh_t eh_from_float(float f) {
  const uint32_t r = eh2_pack(f, 0.f);
  return __ushort_as_half((unsigned short)(r & 0xffffu));
}
__device__ __forceinline__ float eh_to_float(eh_t v) { return __half2float(v); }
__device__ __forceinline__ float2 eh2_unpack(uint32_t w) { return __half22float2(*reinterpret_cast<const __half2*>(&w)); }
#else
typedef __nv_bfloat16 eh_t;
typedef __nv_bfloat162 eh2_t;
#define FRX_EH_PTX "bf16"
__device__ __forceinline__ uint32_t eh2_pack(float lo, float hi) {
  __nv_bfloat162 t = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&t);
}
__device__ __forceinline__ eh_t eh_from_float(float f) { return __float2bfloat16_rn(f); }
__device__ __forceinline__ float eh_to_float(eh_t v) { return __bfloat162float(v); }
__device__ __forceinline__ float2 eh2_unpack(uint32_t w) { return make_float2(__uint_as_float(w << 16), __uint_as_float(w & 0xffff0000u)); }
#endif

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// ---------------------------------------------------------------------------
// Parameter blocks (plain structs passed by value to the kernels)
// ---------------------------------------------------------------------------
// Implicit-GEMM convolution / dense GEMM:  C[M,N] = epi( A[M,K] * W[N,K]^T )
struct GemmP {
  const float* A;      // dense: [M, lda]; conv: NHWC activation
  const float* W;      // [N, K]  (K contiguous; conv K index = (kh*KW+kw)*Cin + ci)
  float* C;            // [M, ldc]
  int M, N, K;
  int lda, ldc;
  int conv;            // 0 = dense, 1 = NHWC gather
  int H, Wd, Cin, OH, OW, KH, KW, stride, pad_t, pad_l;
  const float* gate;   // dense only: per-image per-k multiplier [M/rows_per_img, K] (SE excite)
  int rows_per_img;
  const float* scale;  // per-N: v = v*scale[n] + shift[n]   (folded eval BatchNorm)
  const float* shift;  // per-N: bias when scale == nullptr
  int act;
  const float* res;    // residual added after the activation, [M, ldr]
  int ldr;
  // deterministic split-K (training step: skinny GEMMs whose few tiles would walk a long K serially): the launcher picks
  // the split when a workspace is given; partial tiles go to ws [split][M][N], a second kernel sums them in split order
  // and applies the epilogue
  float* ws;           // nullptr: never split (the inference paths)
  long long ws_floats;
  int splitk, k_chunk; // set by the launcher
};

// Philox4x32-10 (Random123; the generator of curand_Philox4x32_10): counter c, key k -> four 32-bit words
__host__ __device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint2 k) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint64_t p0 = (uint64_t)0xD2511F53u * c.x, p1 = (uint64_t)0xCD9E8D57u * c.z;
    c = make_uint4((uint32_t)(p1 >> 32) ^ c.y ^ k.x, (uint32_t)p1, (uint32_t)(p0 >> 32) ^ c.w ^ k.y, (uint32_t)p0);
    k.x += 0x9E3779B9u;
    k.y += 0xBB67AE85u;
  }
  return c;
}

// One dropout site of the training step.  Element e (its index in the site's logical layout) is kept iff word e % 4 of
// philox4x32_10((e / 4, site, step, rank), (seed_lo, seed_hi)) is >= thresh; kept values are multiplied by scale, dropped
// ones are 0.  step is read from device memory (*step - back), so a CUDA graph of the pass draws new masks on every replay:
// the forward kernels read the counter with back = 0, the backward kernels (after the forward has advanced it) with 1.
struct DropP {
  const uint32_t* step;   // nullptr: the site is off
  uint32_t back;
  uint32_t site, rank;
  uint32_t key_lo, key_hi;
  uint32_t thresh;
  float scale;
};
__device__ __forceinline__ float drop_factor(const DropP& d, long long e) {
  const uint4 r = philox4x32_10(make_uint4((uint32_t)(e >> 2), d.site, *d.step - d.back, d.rank), make_uint2(d.key_lo, d.key_hi));
  const int w = (int)(e & 3);
  const uint32_t u = w == 0 ? r.x : w == 1 ? r.y : w == 2 ? r.z : r.w;
  return u >= d.thresh ? d.scale : 0.f;
}

struct DwP {
  const float* in;     // NHWC [B,H,W,C]
  const float* w;      // [9][C]
  const float* scale;  // [C]
  const float* shift;  // [C]  (conv bias already folded in)
  float* out;          // NHWC [B,OH,OW,C]
  int B, H, Wd, C, OH, OW, stride, pad_t, pad_l, act;
};

struct Seg {           // output column segment of a decoder GEMM
  int n_begin, n_end;
  float* dst;          // element (m, n) -> dst[m*row_stride + slot*slot_stride + (n - n_begin)]
  long long row_stride;
  long long slot_stride;   // multiplied by row_slot[m] when row_slot != nullptr
};

struct DecGemmP {
  const float* A;      // [M, K] row-major (pre-LayerNorm values when ln_g != nullptr)
  const float* Wt;     // [K, N] (N contiguous)
  const float* bias;   // [N]
  int M, N, K, lda;
  int act;
  const float* res;    // [M, ldr] added after the activation
  int ldr;
  const float* ln_g;   // LayerNorm applied to A rows on load (requires K == row width)
  const float* ln_b;
  float* a_norm_out;   // normalised A written back by the n-tile-0 blocks (or nullptr)
  const int* row_slot; // optional per-row slot index for Seg::slot_stride
  int nseg;
  Seg seg[4];
};

struct AttnP {
  const float* q;      // [M, ldq]  query rows (head h at columns h*HD)
  int ldq;
  const float* kcache; // [Bimg, rows_per_img, D]
  const float* vcache;
  int rows_per_img;    // row capacity per image in the cache
  int D;               // model width of the cache rows
  int n_hist;          // number of cached rows attended (when hist_len == nullptr)
  const int* hist_len; // optional per-row history length
  int causal_L;        // > 0: history length of row m is (m % causal_L) + 1 (teacher-forced causal mask)
  const unsigned char* key_mask;  // optional [Bimg, rows_per_img]: 1 = key masked (-inf), e.g. PAD tokens
  const int* chain;    // optional [M, chain_stride] row indices (tree-structured history)
  int chain_stride;
  const float* cur_k;  // optional current key/value row per query [M, ld_cur] (extra last key)
  const float* cur_v;
  int ld_cur;
  int q_per_img;       // query rows per image (1 for incremental decode, L for teacher forcing)
  float temperature;   // scores are DIVIDED by this
  float* out;          // [M, ldo]
  int ldo;
  int M;
  int heads;
};


// best-first "beam" search state (kernels_beam.cu); arrays are [B][cap] unless noted
struct BeamP {
  int B, V, bw, max_seq, T, cap, sos, eos, pad;
  double* hscore; int* hnode; int* hsize;                          // binary heap (heapq order)
  int* nprev; int* ntok; int* nlen; double* nlogp; int* nkv; int* ncount;   // search-tree nodes
  int *num_steps, *done, *endnode, *nexp, *cur_node;               // [B]
  int *cur_tok, *pos, *slot, *active;                              // [B] inputs of the decoder step
  int* chain;                                                      // [B][T] K/V cache rows of the ancestors
  int* n_active;                                                   // [1]
  const float* logits;                                             // [B][V]
  long long* out;                                                  // [B][max_seq]
};

// tcgen05 implicit GEMM (kernels_tc.cu):  C[M,N] = epi( A[M,K] * W[N,K]^T ), bf16 operands
struct TcGemmP {
  const eh_t* A;            // dense [M, lda] or NHWC activation (conv = 1)
  const eh_t* W;            // [N, ldw], K contiguous (conv K index = (kh*KW+kw)*Cin + ci)
  void* C;                  // bf16 or fp32 [M, ldc]
  int M, N, K, lda, ldw, ldc;
  int BN;                   // N tile (multiple of 16, <= 256); 0 = choose
  int stages;               // smem ring depth (set by the launcher)
  int conv, H, Wd, Cin, OH, OW, KW, stride, pad_t, pad_l;
  const eh_t* Wpad; // conv only, optional: weights as [N][KW*KW][64] (channels zero-padded to 64) for the
                             // TMA-im2col path (one filter tap = one 64-wide k-block); nullptr = cp.async gather
  int im2col;               // set by the launcher when the im2col tensor map could be built
  const float* scale;       // per-N folded BatchNorm (v*scale + shift) or nullptr
  const float* shift;       // per-N bias when scale == nullptr
  int act;
  const void* res;          // residual added after the activation ([M, ldr], bf16 or fp32)
  int res_f32, ldr, out_f32;
};

// ids of the tokens the DecodingManager rules single out (dec_sift_embed_kernel)
struct SiftIds { int sos, eos, empty, lbrace, rbrace, underbar; };

// ---------------------------------------------------------------------------
// bf16 persistent decode kernel (kernels_decode_bf16.cu)
// ---------------------------------------------------------------------------
constexpr int DEC_CLUSTER = 8;   // CTAs per cluster
constexpr int DEC_IMG = 8;       // images per cluster (rows 0..7 of the mma.m16n8k16 tile)
constexpr int DEC_FMAX = 1024;   // decoder filter_dim the kernel is specialised for
constexpr int DEC_TMAX = 500;    // max decode steps of the cluster kernel = length of the 1-D positional table (PositionEncoder1D max_len, EfficientSATRN.py:408); nothing in the kernel is sized by it
constexpr int DEC_MAX_CLUSTERS = 32;  // clusters per launch; 33 8-CTA clusters are co-resident at 2 CTAs/SM on B200

struct DecClusterLayer {
  const uint4 *w_o, *w_q2, *w_o2, *w_f0, *w_f1, *w_next;   // fragment-packed bf16, per-CTA blocks
  const float *b_o, *b_q2, *b_o2, *b_f0, *b_f1, *b_next;   // fp32 biases, natural column order
  const float *ln1_g, *ln1_b, *ln2_g, *ln2_b, *ln3_g, *ln3_b;
};

struct DecClusterP {
  int B, steps, T, L, V, S, sos;
  int img_base;                  // first image of this launch (set by the launcher)
  const uint4* w_first;          // layer-0 q|k|v
  const float* b_first;
  DecClusterLayer layer[4];
  const float* emb;              // [V+1][D] fp32
  const float* pe;               // [500][D] fp32
  __nv_bfloat16* kself;          // [L][B][H][T][32]
  __nv_bfloat16* vself;
  const __nv_bfloat16* kcross;   // [L][B][H][S][32]
  const __nv_bfloat16* vcross;
  float* logits;                 // [B][steps][V] or nullptr
  long long* tokens;             // [B][steps] or nullptr
  const long long* forced;       // [B][steps] or nullptr
  // "step mode" (step_forward / ensemble / best-first search): one launch = `steps` steps (normally 1) that CONTINUE a
  // history instead of starting at <SOS>.  All nullptr = a greedy decode from position 0.
  const int* hist_len;           // [B] keys already cached for the image = position of this launch's first step
  const int* chain;              // [B][T] cache rows of those keys in attention order (ancestor chain); nullptr = rows 0..n-1
  const int* slot;               // [B] cache row that receives the first step's K/V; nullptr = hist_len[b] (+ step)
  const int* first_tok32;        // [B] token fed at the first step (int32), or
  const long long* first_tok64;  // [B] the same as int64; both nullptr = <SOS>
  // rule-constrained decoding (DecodingManager.sift, postprocessing/postprocessing.py:193-391): per-class rule tables;
  // sift_flags != nullptr -> the pick stage soft-maxes, black-lists and takes the constrained arg-max, `logits` receives
  // the masked probabilities (EfficientSATRN.py:553-555) and the MemoryNode state lives in the pick warps' registers
  const int* sift_flags;
  const int* sift_limit;
  SiftIds sift_ids;
  long long* prof;               // optional [16] per-stage cycle totals (cluster 0, CTA 0, thread 0)
  // stop-at-<EOS> instantiations (FRX_DEC_EOS): each of a cluster's rows decodes one image until it emits `eos` (forced:
  // until forced[b][t] == eos) or reaches `steps`, writes lengths[b] = steps decoded, and takes the next image from the
  // zeroed counter *work.  The self K/V caches are indexed by slot (cluster * 8 + row) instead of by image.
  int* lengths;                  // [B] int32
  int* work;                     // images handed out so far (zero before the launch)
  int eos;
};

}  // namespace frx
