// kernels_decode_bf16.cu -- the whole greedy decode loop as ONE persistent kernel.
//
// A thread-block CLUSTER of 8 CTAs owns 8 images for all steps; CTA r of the cluster owns
// attention HEAD r of those images and 1/8 of the output columns of every other linear layer:
//   * q|k|v of head r are computed by CTA r (the 96 columns of the fused projection that belong to the
//     head) and consumed by CTA r's own attention warps (warp w <-> image w) straight from shared memory:
//     q, k, v never cross a CTA boundary, and the K/V cache of (image, head r) is written and read by one
//     CTA only, so no cross-CTA global-memory visibility is needed anywhere;
//   * what does cross CTA boundaries is all-gathered through distributed shared memory with st.async: the
//     attention outputs (2x per layer), the pre-LayerNorm rows (3x) and the FFN hidden row (1x) = 6
//     exchanges per layer + the logits = 19 per step.  Every store completes transaction bytes on the
//     DESTINATION CTA's mbarrier; a stage is over for a CTA when the bytes it expects have landed -- no
//     cluster barrier, no fence;
//   * linear layers run on mma.sync.m16n8k16 (bf16 -> fp32) with the weights streamed from L2 in
//     B-fragment order (packed on the host).  Every warp requests the weight fragments of its share of a
//     stage before the wait that precedes the stage (weights are static), so a stage costs one L2 round
//     trip at most; every stage is K-split over two warps, the partial fragments meet in shared memory and
//     the epilogue works on 8-column row pieces so that all DSMEM / global stores are 16 bytes wide;
//   * attention of (image w, head r) is one warp on the tensor cores (q replicated over the MMA rows), K/V
//     rows staged global -> shared one or two 32-key blocks ahead and turned into B fragments with ldmatrix /
//     ldmatrix.trans.  The caches keep every row's 16-byte chunks pre-swizzled in HBM, so a block of a contiguous
//     history is one contiguous piece: the two-block-ring geometry fetches it with ONE bulk copy per operand
//     (cp.async.bulk on a per-slot mbarrier) and requests the next phase's first blocks as soon as the ring is idle;
//     the other geometries (and ancestor-chain histories) use per-lane cp.async;
//   * work that nobody waits for in this step -- the K/V cache rows of the layer OUTPUT (SURVEY F3: the
//     reference caches layer outputs) -- runs between a stage's stores and its wait.
// LayerNorm / residual are recomputed redundantly per CTA on the gathered rows (cheaper than another
// exchange).  tcgen05 is not used here on purpose: M is 8..16 rows per cluster (DESIGN.md 4.1).
//
// Implements the recurrence of SURVEY App. A.4 (networks/EfficientSATRN.py:374-397, :539-558): cached
// layer OUTPUTS, current layer INPUT as the last key, scores divided by sqrt(d_model), post-LN, ReLU
// after both FFN linears.
#include <cooperative_groups.h>
#include <cstdio>
#include <cstdlib>

#include "common.cuh"
#include "kernels.h"

namespace cg = cooperative_groups;

namespace frx {

namespace {

// The kernel is specialised at compile time for one decoder geometry; the default is EfficientSATRN's (hidden 256,
// 8 heads, filter 1024 -> clusters of 8 CTAs).  kernels_decode_bf16_d128.cu re-includes this file for LiteSATRN's
// (hidden 128, 4 heads, filter 512 -> clusters of 4).  Head width is 32 and one CTA owns one head in both.
#ifndef FRX_DEC_D
#define FRX_DEC_D 256
#define FRX_DEC_FF 1024
#define FRX_DEC_NAME(x) x
#endif
#ifndef FRX_DEC_HPC
#define FRX_DEC_HPC 1            // heads per CTA; 2 = kernels_decode_bf16_p2.cu: clusters of 4 CTAs x 16 warps, one CTA per SM
#endif
#ifndef FRX_DEC_HD
#define FRX_DEC_HD 32            // head width (64: kernels_decode_bf16_d512.cu, the SwinTRN decoder)
#endif
constexpr int D = FRX_DEC_D;     // decoder width
constexpr int HD = FRX_DEC_HD;
constexpr int H = D / HD;        // heads
#ifndef FRX_DEC_KVDEPTH
#define FRX_DEC_KVDEPTH 1        // K/V staging blocks per warp (blocks in flight ahead of the one being reduced)
#endif
constexpr int HPC = FRX_DEC_HPC;
constexpr int KVD = FRX_DEC_KVDEPTH;
#ifndef FRX_DEC_KVBULK
#define FRX_DEC_KVBULK (FRX_DEC_KVDEPTH >= 2)   // contiguous K/V histories by bulk copies: pays with two blocks in flight (see kv_request_bulk)
#endif
constexpr bool KV_BULK = FRX_DEC_KVBULK;
#ifndef FRX_DEC_EARLYPRIME
#define FRX_DEC_EARLYPRIME FRX_DEC_KVBULK   // request the next attention phase's first K/V blocks as soon as the ring is idle (measured: pays with the bulk-copy ring only)
#endif
constexpr bool EARLY_PRIME = FRX_DEC_EARLYPRIME;
#ifdef FRX_DEC_EOS
constexpr bool EOS = true;       // rows stop at <EOS> and are refilled with the next image (kernels_decode_bf16*_eos.cu)
#else
constexpr bool EOS = false;
#endif
constexpr int CL = H / HPC;      // CTAs per cluster
constexpr int FF = FRX_DEC_FF;
constexpr int VP = 256;          // vocabulary columns, padded
constexpr int SW = D / CL;       // columns of D per CTA (its heads)
constexpr int FS = FF / CL;      // columns of the FFN hidden row per CTA
constexpr int NTS = SW / 8, NTA = 3 * NTS, NTC = 2 * NTS, NTE = FS / 8;  // tiles: slice, q|k|v, K|V cache rows, FFN0
constexpr int NG = VP / CL / 8;  // generator tiles per CTA
static_assert(SW == HD * HPC && CL <= 8 && (8 % CL) == 0 && FS % 8 == 0, "column slices");
constexpr int APAD = 8;          // bf16 padding of the A-operand rows (conflict-free ldmatrix)
constexpr int FPAD = 4;          // fp32 padding of rows that are accessed 16 bytes per lane, 8 rows at a time
constexpr int NIMG = DEC_IMG;    // images per cluster = warps per CTA (warp w <-> image w)
constexpr int NWARP = NIMG * HPC; // warp w <-> (image w % NIMG, head-of-this-CTA w / NIMG)
constexpr int NTHR = NWARP * 32;
constexpr int RED_FLOATS = 2 * (NTE > NTA ? NTE : NTA) * 64;  // K-split reduction region: KS * NT * 32 lanes * 2 floats, widest stage
static_assert(NIMG == 8, "the kernel maps MMA rows 0..7 to the cluster's images");

__device__ __forceinline__ void mma_bf16(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};\n"
      : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}

__device__ __forceinline__ uint64_t make_evict_last_policy() {
  uint64_t pol;
  asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;\n" : "=l"(pol));
  return pol;
}

__device__ __forceinline__ uint4 ldg_weights(const uint4* p, uint64_t pol) {
  uint4 v;  // weights are re-read every step by every cluster: ask L2 to keep them
  asm("ld.global.nc.L1::no_allocate.L2::cache_hint.v4.u32 {%0,%1,%2,%3}, [%4], %5;\n"
      : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p), "l"(pol));
  return v;
}

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ uint32_t pack_bf16(float lo, float hi) {
  __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&v);
}

__device__ __forceinline__ void unpack8(const uint4& u, float (&f)[8]) {
  const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    f[2 * i] = __uint_as_float(w[i] << 16);
    f[2 * i + 1] = __uint_as_float(w[i] & 0xffff0000u);
  }
}

struct Smem {
  // row strides are padded by 16 bytes wherever a quarter-warp touches 8 rows with 16-byte accesses
  float xres[NIMG][D + FPAD];           // residual stream (fp32), full rows in every CTA
  float pre[NIMG][D + FPAD];            // gathered pre-LayerNorm rows
  __nv_bfloat16 abf[NIMG][D + APAD];    // A operand: LayerNorm output / embedded input
  __nv_bfloat16 obf[NIMG][D + APAD];    // A operand: gathered attention outputs (all heads)
  __nv_bfloat16 abf2[NIMG][FF + APAD];  // A operand: gathered FFN hidden row (also the fp32 logits view)
  float red[2][RED_FLOATS];             // K-split partial fragments (two alternating regions)
  float qh[HPC][NIMG][HD + FPAD];            // q of this CTA's head(s)
  __nv_bfloat16 kcur[HPC][NIMG][HD + APAD];  // k, v of the current layer input (the extra "current" key)
  __nv_bfloat16 vcur[HPC][NIMG][HD + APAD];
  __nv_bfloat16 kvst[NWARP][KVD][2][32][HD]; // per-warp ring of KVD staged 32-key K/V blocks (KVStage)
  long long prof[16];
  int4 sift[NIMG];                      // DecodingManager: MemoryNode of each row {current token, run length, #'{', #'}'}
  unsigned long long bar[2];            // stage mbarriers (alternate by stage parity)
  unsigned long long kvbar[NWARP][KVD]; // per-warp mbarriers of the K/V ring slots (bulk copies of contiguous histories)
  DecClusterLayer lw[4];                // per-layer pointers (dynamic indexing of kernel params would spill them)
};
// Per-row state of the stop-at-<EOS> instantiations, in shared memory behind Smem (the two-heads geometry has no
// registers to spare for it).
struct EosRows {
  int img[NIMG];                        // image each row decodes (-1: idle, no work left)
  int pos[NIMG];                        // its position = the step it is at
  int done[NIMG];                       // the row finished its image at this step
  int left[NIMG];                       // history length of the image a refilled row left (its early-primed K/V blocks)
  int claim[8];                         // claim[c]: what CTA c sent in this step's refill exchange (rank 0: first image)
};
constexpr size_t SMEM_BYTES = sizeof(Smem) + (EOS ? sizeof(EosRows) : 0);
static_assert(!(EOS && EARLY_PRIME) || KV_BULK, "a refilled row drains the early-primed blocks on the ring's mbarriers");

// ---------------------------------------------------------------------------
// GEMM stage: out[8 images, NT*8 columns of this CTA] = A[8, K] * W^T; A bf16 in smem (rows 8..15 of the
// MMA tile alias rows 0..7), W fragment-packed [tile][K/32][32 lanes] uint4.  The K range is split over
// KS warps (warp w: k-slice w % KS, tiles (w / KS) + j*TG); the partial fragments meet in shared memory and
// the epilogue runs on (tile, row) units of 8 consecutive columns so that everything it stores is 16 bytes
// wide: epi(tile, row, v[8], sub) with sub in [0, NTHR / (NT*8)) distinguishing the threads that share a unit
// (they split the destinations of an all-gather between them).
// ---------------------------------------------------------------------------
template <int NT, int KP, int KS>
struct GC {
  static constexpr int NW = NTHR / 32, TG = NW / KS, TPW = NT / TG, KPW = KP / KS, TOT = TPW * KPW;
  static constexpr int UNITS = NT * 8, NSUB = NTHR / UNITS;
  static_assert(NW % KS == 0 && NT % TG == 0 && KP % KS == 0 && NSUB >= 1, "bad GEMM split");
  static_assert(KS * NT * 64 <= RED_FLOATS, "reduction region too small");
};

template <int N>
struct WPre { uint4 w[N > 0 ? N : 1]; };

template <int NT, int KP, int KS, int PF>
__device__ __forceinline__ WPre<PF> prefetch_w(const uint4* __restrict__ Wp, uint64_t pol) {
  using C = GC<NT, KP, KS>;
  WPre<PF> pre;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int ks = warp % KS, tg = warp / KS;
#pragma unroll
  for (int idx = 0; idx < PF; ++idx) {
    const int kk = idx / C::TPW, j = idx % C::TPW;
    pre.w[idx] = ldg_weights(Wp + ((size_t)(tg + j * C::TG) * KP + ks * C::KPW + kk) * 32 + lane, pol);
  }
  return pre;
}

template <int NT, int KP, int KS, int PF, typename Epi>
__device__ __forceinline__ void gemm2(float* __restrict__ red, const __nv_bfloat16* A, int lda,
                                      const uint4* __restrict__ Wp, uint64_t pol, const WPre<PF>& pre, Epi epi) {
  using C = GC<NT, KP, KS>;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int ks = warp % KS, tg = warp / KS;
  // A fragments of two k16 steps with two ldmatrix.x4: lane -> row address of matrix (lane >> 3):
  // {rows 0-7, k lo}, {rows 8-15, k lo}, {rows 0-7, k hi}, {rows 8-15, k hi}; rows 8-15 alias rows 0-7.
  const uint32_t a_lane = smem_u32(A + (lane & 7) * lda + ((lane >> 4) & 1) * 8);
  float acc[C::TPW][2][4];
#pragma unroll
  for (int j = 0; j < C::TPW; ++j)
#pragma unroll
    for (int h = 0; h < 2; ++h)
#pragma unroll
      for (int e = 0; e < 4; ++e) acc[j][h][e] = 0.f;
  auto wload = [&](int kk, int j) {
    return ldg_weights(Wp + ((size_t)(tg + j * C::TG) * KP + ks * C::KPW + kk) * 32 + lane, pol);
  };
  auto kstep = [&](int kk, const uint4* wk) {
    const uint32_t addr = a_lane + (uint32_t)(ks * C::KPW + kk) * 64u;  // 32 bf16 per k-pair
    uint32_t a0[4], a1[4];
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];\n"
                 : "=r"(a0[0]), "=r"(a0[1]), "=r"(a0[2]), "=r"(a0[3]) : "r"(addr));
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];\n"
                 : "=r"(a1[0]), "=r"(a1[1]), "=r"(a1[2]), "=r"(a1[3]) : "r"(addr + 32u));
#pragma unroll
    for (int j = 0; j < C::TPW; ++j) {
      mma_bf16(acc[j][0], a0, wk[j].x, wk[j].y);
      mma_bf16(acc[j][1], a1, wk[j].z, wk[j].w);
    }
  };
  if constexpr (C::TOT <= 16) {
    // the warp's whole share of the stage's weights in registers (requested up front: one L2 round trip)
    uint4 w[C::TOT];
#pragma unroll
    for (int idx = 0; idx < C::TOT; ++idx) {
      const int kk = idx / C::TPW, j = idx % C::TPW;
      if (idx < PF) w[idx] = pre.w[idx];
      else w[idx] = wload(kk, j);
    }
#pragma unroll
    for (int kk = 0; kk < C::KPW; ++kk) kstep(kk, &w[kk * C::TPW]);
  } else {
    // wide stages (512-wide decoder): stream the fragments two k-pairs ahead through a register ring
    static_assert(PF == 0 || PF == C::TPW, "streaming stages prefetch exactly their first k-pair");
    constexpr int RING = 3;
    uint4 w[RING][C::TPW];
#pragma unroll
    for (int r = 0; r < RING - 1; ++r)
#pragma unroll
      for (int j = 0; j < C::TPW; ++j) {
        if (r < C::KPW) w[r][j] = (PF > 0 && r == 0) ? pre.w[j] : wload(r, j);
      }
#pragma unroll
    for (int kk = 0; kk < C::KPW; ++kk) {
      if (kk + RING - 1 < C::KPW) {
#pragma unroll
        for (int j = 0; j < C::TPW; ++j) w[(kk + RING - 1) % RING][j] = wload(kk + RING - 1, j);
      }
      kstep(kk, w[kk % RING]);
    }
  }
  // partial fragments -> red[ks][tile][lane] (float2: row lane>>2, columns (lane&3)*2 + {0,1})
#pragma unroll
  for (int j = 0; j < C::TPW; ++j)
    *reinterpret_cast<float2*>(red + ((size_t)(ks * NT + tg + j * C::TG) * 32 + lane) * 2) =
        make_float2(acc[j][0][0] + acc[j][1][0], acc[j][0][1] + acc[j][1][1]);
  __syncthreads();
  if (threadIdx.x < C::UNITS * C::NSUB) {
    const int u = threadIdx.x % C::UNITS, sub = threadIdx.x / C::UNITS;
    const int tile = u >> 3, row = u & 7;
    float v[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) v[i] = 0.f;
#pragma unroll
    for (int k2 = 0; k2 < KS; ++k2) {
      const float4* src = reinterpret_cast<const float4*>(red + ((size_t)(k2 * NT + tile) * 32 + row * 4) * 2);
      const float4 lo = src[0], hi = src[1];
      v[0] += lo.x; v[1] += lo.y; v[2] += lo.z; v[3] += lo.w;
      v[4] += hi.x; v[5] += hi.y; v[6] += hi.z; v[7] += hi.w;
    }
    epi(tile, row, v, sub);
  }
}

// ---- DSMEM all-gather with st.async + mbarrier transaction counting ------------------
__device__ __forceinline__ uint32_t mapa_u32(uint32_t addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;\n" : "=r"(r) : "r"(addr), "r"(rank));
  return r;
}
__device__ __forceinline__ void st_async_b32(uint32_t raddr, uint32_t v, uint32_t rbar) {
  asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.b32 [%0], %1, [%2];\n" ::"r"(raddr), "r"(v), "r"(rbar) : "memory");
}
__device__ __forceinline__ void st_async_v4(uint32_t raddr, uint4 v, uint32_t rbar) {
  asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.v4.b32 [%0], {%1, %2, %3, %4}, [%5];\n" ::"r"(raddr), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w), "r"(rbar) : "memory");
}
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;\n" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"(bar), "r"(bytes) : "memory");
}
// Bounded spin: a byte-accounting bug traps (error reaches the host) instead of hanging the GPU.
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok = 0;
#ifndef FRX_DEC_SPINLIMIT
#define FRX_DEC_SPINLIMIT (1ll << 26)
#endif
#pragma unroll 1
  for (long long spins = 0; spins < FRX_DEC_SPINLIMIT; ++spins) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n" : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
    if (ok) return;
  }
  __trap();
}


struct LnParams { float g[D / 32], b[D / 32]; };
__device__ __forceinline__ LnParams load_ln(const float* __restrict__ g, const float* __restrict__ b) {
  LnParams o;  // issued BEFORE the stage wait so the load latency overlaps it
  const int lane = threadIdx.x & 31;
#pragma unroll
  for (int i = 0; i < D / 32; ++i) { o.g[i] = __ldg(g + i * 32 + lane); o.b[i] = __ldg(b + i * 32 + lane); }
  return o;
}

// LayerNorm of the gathered rows: warp w <-> row w (every CTA does all rows).  Mean and centred second
// moment are taken around the lane's own first element (a shift that keeps the single-pass form
// var = E[(x-s)^2] - (E[x-s])^2 well conditioned) so one butterfly carries both sums.
__device__ __forceinline__ void layernorm_rows(Smem& s, const LnParams& P) {
  const int row = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (row >= NIMG) return;  // with more than one head per CTA only the first NIMG warps own a row
  float v[D / 32];
#pragma unroll
  for (int i = 0; i < D / 32; ++i) v[i] = s.pre[row][i * 32 + lane];
  const float shift = __shfl_sync(0xffffffffu, v[0], 0);
  float s1 = 0.f, s2 = 0.f;
#pragma unroll
  for (int i = 0; i < D / 32; ++i) { const float d = v[i] - shift; s1 += d; s2 = fmaf(d, d, s2); }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    s1 += __shfl_xor_sync(0xffffffffu, s1, o);
    s2 += __shfl_xor_sync(0xffffffffu, s2, o);
  }
  const float md = s1 * (1.f / D);
  const float mean = shift + md;
  const float rstd = rsqrtf(fmaxf(s2 * (1.f / D) - md * md, 0.f) + 1e-5f);
#pragma unroll
  for (int i = 0; i < D / 32; ++i) {
    const int c = i * 32 + lane;
    const float o = (v[i] - mean) * rstd * P.g[i] + P.b[i];
    s.xres[row][c] = o;
    s.abf[row][c] = __float2bfloat16_rn(o);
  }
}

// ---------------------------------------------------------------------------
// Attention of one (image, head) pair by one warp on the tensor cores, single pass (online softmax),
// 32 keys per iteration.  The query is one row, so the MMA tile carries it in rows 0..7 (replicated) and
// nothing in rows 8..15; what the tensor core buys here is instruction count (16 HMMA + ~100 other
// instructions per 32 keys instead of ~260 FFMA/shuffle instructions) in an issue-bound phase.
//   * K/V rows ([key][32] bf16, 64 B) travel global -> shared with cp.async (16 B per lane, 512 contiguous
//     bytes per instruction, zero-fill past the history), so a block can be requested long before it is
//     needed without holding registers: block 0 is requested BEFORE the projection GEMM that produces q,
//     block i+1 while block i is being reduced;
//   * B fragments come from shared memory with ldmatrix (K: plain, V: .trans); rows are XOR-swizzled by
//     16-byte chunk so that both the cp.async writes and the ldmatrix reads are bank-conflict-free;
//   * after the loop the extra "current input" key of the reference recurrence (SURVEY F3) is merged.
// Lane (gid, tig) returns dims 8 nt + 2 tig + {0, 1}, nt = 0..3, in o[2 nt + {0, 1}]; the eight gid groups
// hold identical copies.
// ---------------------------------------------------------------------------
struct KVStage { __nv_bfloat16 k[32][HD], v[32][HD]; };  // one 32-key block of one warp (4 KB)

// row = key (HD * 2 bytes), chunk = 16-byte piece of it; XOR swizzle of the chunk position inside the row so that the
// staging writes and the ldmatrix reads are conflict-free.  The K/V caches in HBM keep every row in the SAME permuted
// chunk order (kv_perm of the cache row; the permutation has period 8 in the row index and blocks start at multiples of
// 32), so a 32-key block of a contiguous history is one contiguous, already-swizzled piece of memory: one bulk copy.
__device__ __forceinline__ int kv_perm(int row) {
  if constexpr (HD == 32) return (row >> 1) & 3;
  else return row & (HD / 8 - 1);
}
__device__ __forceinline__ uint32_t kv_swz(int row, int chunk) { return (uint32_t)(row * (HD * 2) + ((chunk ^ kv_perm(row)) << 4)); }

__device__ __forceinline__ void kv_request(KVStage& st, const __nv_bfloat16* __restrict__ Kc, const __nv_bfloat16* __restrict__ Vc,
                                           int kb, int n_hist, const int* __restrict__ chain) {
  // one commit group per call, EMPTY when the block lies past the history: the consumer counts groups.  chain != nullptr:
  // key j of the history lives in cache row chain[j] (the ancestors of a search-tree node), otherwise in row j.
  if (kb < n_hist) {
    const int lane = threadIdx.x & 31;
    const uint32_t ks = smem_u32(&st.k[0][0]), vs = smem_u32(&st.v[0][0]);
#pragma unroll
    for (int i = 0; i < HD / 8; ++i) {
      const int id = lane + 32 * i, row = id / (HD / 8), chunk = id % (HD / 8);
      const int key = kb + row;
      const uint32_t bytes = key < n_hist ? 16u : 0u;   // zero-fill past the history (also keeps V finite)
      int src = key < n_hist ? key : 0;
      if (chain) src = __ldg(chain + src);
      const size_t off = (size_t)src * HD + ((chunk ^ kv_perm(src)) << 3);   // the cache row keeps its chunks permuted
      asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;\n" ::"r"(ks + kv_swz(row, chunk)), "l"(Kc + off), "r"(bytes) : "memory");
      asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;\n" ::"r"(vs + kv_swz(row, chunk)), "l"(Vc + off), "r"(bytes) : "memory");
    }
  }
  asm volatile("cp.async.commit_group;\n" ::: "memory");
}
// Contiguous history (no ancestor chain): the block is ONE bulk copy per operand (cp.async.bulk, issued by lane 0,
// completing on the warp's mbarrier of that ring slot) instead of 2 * HD / 8 cp.async per lane -- the per-lane copies and
// their address arithmetic were where the attention phase stalled (mio_throttle / long_scoreboard on the LDGSTS).  Only
// the valid rows travel; the rows behind them keep older (finite) K/V data or the zeros of the kernel prologue, and their
// probabilities are exactly 0.  Blocks past the history are neither requested nor waited for.
__device__ __forceinline__ void kv_request_bulk(KVStage& st, uint32_t bar, const __nv_bfloat16* __restrict__ Kc,
                                                const __nv_bfloat16* __restrict__ Vc, int kb, int n_hist) {
  if (kb < n_hist && (threadIdx.x & 31) == 0) {
    const int rows = n_hist - kb < 32 ? n_hist - kb : 32;
    const uint32_t bytes = (uint32_t)rows * (HD * 2);
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"(bar), "r"(2u * bytes) : "memory");
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];\n"
                 ::"r"(smem_u32(&st.k[0][0])), "l"(Kc + (size_t)kb * HD), "r"(bytes), "r"(bar) : "memory");
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];\n"
                 ::"r"(smem_u32(&st.v[0][0])), "l"(Vc + (size_t)kb * HD), "r"(bytes), "r"(bar) : "memory");
  }
}
// Request the first KVD blocks of a history into the warp's ring (in block order; with an ancestor chain: KVD commit
// groups of per-lane cp.async, otherwise bulk copies on the ring slots' mbarriers kvbar, kvbar + 8, ...).
__device__ __forceinline__ void kv_prime(KVStage* ring, const __nv_bfloat16* __restrict__ Kc, const __nv_bfloat16* __restrict__ Vc, int n_hist,
                                         const int* __restrict__ chain, uint32_t kvbar) {
  if (!KV_BULK || chain) {
#pragma unroll
    for (int d = 0; d < KVD; ++d) kv_request(ring[d], Kc, Vc, 32 * d, n_hist, chain);
  } else {
#pragma unroll
    for (int d = 0; d < KVD; ++d) kv_request_bulk(ring[d], kvbar + 8u * d, Kc, Vc, 32 * d, n_hist);
  }
}

__device__ __forceinline__ float ex2f(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;\n" : "=f"(y) : "f"(x));
  return y;
}

// The history must have been primed with kv_prime(ring, Kc, Vc, n_hist): block i lives in ring[i % KVD] and is
// complete once at most KVD - 1 younger commit groups are pending (cp.async path) / its slot's mbarrier phase has
// completed (bulk path); its buffer is re-used for block i + KVD as soon as its fragments are in registers, so KVD
// blocks are in flight while one is being reduced.
// The phase is ISSUE-bound with 16 warps per SM (~300 executed instructions per warp and 32-key block against 16 HMMA),
// so the loop body is kept lean: q is pre-multiplied by qscale = log2(e) / sqrt(d_model) when it is packed (scores come
// out of the MMA in exp2 units: no per-score scaling, ex2 instead of exp), the key mask runs in the one partial block
// only, the running-maximum rescale only when the maximum moved (warp-uniform: the eight MMA rows are replicas), and the
// ldmatrix offsets are lane constants.  BULK selects the staging path at compile time (false: cp.async, also the only
// path for ancestor chains).
template <bool BULK>
__device__ __forceinline__ void attend_mma(KVStage* ring, const float* __restrict__ q, const __nv_bfloat16* __restrict__ Kc,
                                           const __nv_bfloat16* __restrict__ Vc, int n_hist, const int* __restrict__ chain,
                                           uint32_t kvbar, uint32_t& kvphase, const __nv_bfloat16* __restrict__ kx,
                                           const __nv_bfloat16* __restrict__ vx, float qscale,
                                           float (&o)[HD / 4], long long* pw = nullptr) {
  constexpr int NK = HD / 16;   // k16 steps of q . k
  constexpr int ND = HD / 8;    // 8-wide n-tiles of the output row
  const int lane = threadIdx.x & 31, tig = lane & 3;
  uint32_t aq[NK][4];
#pragma unroll
  for (int ks = 0; ks < NK; ++ks) {
    const float2 qa = *reinterpret_cast<const float2*>(q + 16 * ks + 2 * tig), qb = *reinterpret_cast<const float2*>(q + 16 * ks + 8 + 2 * tig);
    aq[ks][0] = pack_bf16(qa.x * qscale, qa.y * qscale); aq[ks][1] = 0u;
    aq[ks][2] = pack_bf16(qb.x * qscale, qb.y * qscale); aq[ks][3] = 0u;
  }
  float m = -INFINITY, l = 0.f;
  float acc[ND][4];
#pragma unroll
  for (int nt = 0; nt < ND; ++nt)
#pragma unroll
    for (int e = 0; e < 4; ++e) acc[nt][e] = 0.f;
  const int lrow = lane & 7, lmat = lane >> 3;
  // ldmatrix lane offsets inside a staged block (the swizzle term has period 8 in the key index, so tile j / k-step ks2
  // add a constant): K tile j = keys 8j..8j+7, four 8-dim chunks per x4; V k-step ks2, n-tile pair np
  uint32_t koff[ND / 4], voff[ND / 2];
#pragma unroll
  for (int c4 = 0; c4 < ND / 4; ++c4) koff[c4] = kv_swz(lrow, 4 * c4 + lmat);
#pragma unroll
  for (int np = 0; np < ND / 2; ++np) voff[np] = kv_swz((lmat & 1) * 8 + lrow, 2 * np + (lmat >> 1));
  int slot = 0;
  for (int kb = 0; kb < n_hist; kb += 32) {
    KVStage& st = ring[slot];
    const int cur = slot;   // ring slot of this block
    slot = slot + 1 == KVD ? 0 : slot + 1;
    const uint32_t ks = smem_u32(&st.k[0][0]), vs = smem_u32(&st.v[0][0]);
    long long tw = 0;
    if (pw) tw = clock64();
    if (!BULK) {
      asm volatile("cp.async.wait_group %0;\n" ::"n"(KVD - 1) : "memory");
    } else {
      mbar_wait(kvbar + 8u * cur, (kvphase >> cur) & 1u);
      kvphase ^= 1u << cur;
    }
    if (pw) { const long long tn = clock64(); pw[0] += tn - tw; pw[1] += 1; tw = tn; }   // profiler: cycles spent waiting for K/V blocks, blocks reduced
    __syncwarp();
    uint32_t kf[4][ND], vf[2][ND / 2][4];
#pragma unroll
    for (int j = 0; j < 4; ++j)     // score tile j: keys 8j..8j+7; one ldmatrix.x4 = four 8-dim chunks of those keys
#pragma unroll
      for (int c4 = 0; c4 < ND / 4; ++c4)
        asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];\n"
                     : "=r"(kf[j][4 * c4 + 0]), "=r"(kf[j][4 * c4 + 1]), "=r"(kf[j][4 * c4 + 2]), "=r"(kf[j][4 * c4 + 3])
                     : "r"(ks + koff[c4] + (uint32_t)(j * 8 * HD * 2)));
#pragma unroll
    for (int ks2 = 0; ks2 < 2; ++ks2)        // 16-key k-step of P . V
#pragma unroll
      for (int np = 0; np < ND / 2; ++np)    // pair of 8-dim n-tiles
        asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];\n"
                     : "=r"(vf[ks2][np][0]), "=r"(vf[ks2][np][1]), "=r"(vf[ks2][np][2]), "=r"(vf[ks2][np][3])
                     : "r"(vs + voff[np] + (uint32_t)(ks2 * 16 * HD * 2)));
    __syncwarp();
    if (!BULK) kv_request(st, Kc, Vc, kb + 32 * KVD, n_hist, chain);
    else kv_request_bulk(st, kvbar + 8u * cur, Kc, Vc, kb + 32 * KVD, n_hist);
    if (pw) { const long long tn = clock64(); pw[2] += tn - tw; tw = tn; }   // fragments loaded, next block requested
    float sc[4][4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
#pragma unroll
      for (int e = 0; e < 4; ++e) sc[j][e] = 0.f;
#pragma unroll
      for (int k2 = 0; k2 < NK; ++k2) mma_bf16(sc[j], aq[k2], kf[j][2 * k2], kf[j][2 * k2 + 1]);
    }
    // (the branches pay in the issue-bound two-heads-per-CTA geometry; with 8 warps per SM the phase is latency-bound and
    // the same arithmetic runs straight-line: masking every block, scaling by ex2(0) = 1 when the maximum did not move)
    if (!BULK || kb + 32 > n_hist) {   // the one partial block of a history: keys past it score -inf
#pragma unroll
      for (int j = 0; j < 4; ++j)
#pragma unroll
        for (int e = 0; e < 2; ++e)
          if (kb + 8 * j + 2 * tig + e >= n_hist) sc[j][e] = -INFINITY;
    }
    float cm = fmaxf(fmaxf(fmaxf(sc[0][0], sc[0][1]), fmaxf(sc[1][0], sc[1][1])), fmaxf(fmaxf(sc[2][0], sc[2][1]), fmaxf(sc[3][0], sc[3][1])));
    cm = fmaxf(cm, __shfl_xor_sync(0xffffffffu, cm, 1));
    cm = fmaxf(cm, __shfl_xor_sync(0xffffffffu, cm, 2));
    cm = fmaxf(cm, m);
    if (!BULK || cm > m) {    // the running maximum moved: rescale what has been accumulated (ex2(-inf) = 0 the first time)
      const float scale = ex2f(m - cm);
      m = cm;
      l *= scale;
#pragma unroll
      for (int nt = 0; nt < ND; ++nt) { acc[nt][0] *= scale; acc[nt][1] *= scale; }
    }
    if (pw) { const long long tn = clock64(); pw[3] += tn - tw; tw = tn; }   // scores, running maximum
    float pr[4][2];
#pragma unroll
    for (int j = 0; j < 4; ++j)
#pragma unroll
      for (int e = 0; e < 2; ++e) pr[j][e] = ex2f(sc[j][e] - m);
    l += ((pr[0][0] + pr[0][1]) + (pr[1][0] + pr[1][1])) + ((pr[2][0] + pr[2][1]) + (pr[3][0] + pr[3][1]));
#pragma unroll
    for (int ks2 = 0; ks2 < 2; ++ks2) {  // 16 keys per k-step: score tiles 2 ks2 (k lo) and 2 ks2 + 1 (k hi)
      const uint32_t ap[4] = {pack_bf16(pr[2 * ks2][0], pr[2 * ks2][1]), 0u, pack_bf16(pr[2 * ks2 + 1][0], pr[2 * ks2 + 1][1]), 0u};
#pragma unroll
      for (int np = 0; np < ND / 2; ++np) {
        mma_bf16(acc[2 * np], ap, vf[ks2][np][0], vf[ks2][np][1]);
        mma_bf16(acc[2 * np + 1], ap, vf[ks2][np][2], vf[ks2][np][3]);
      }
    }
    if (pw) pw[4] += clock64() - tw;   // probabilities, P . V issued
  }
  l += __shfl_xor_sync(0xffffffffu, l, 1);
  l += __shfl_xor_sync(0xffffffffu, l, 2);
  if (kx) {
    constexpr int DPT = HD / 4;   // dims of the "current input" key per lane of a quad
    float part = 0.f;
#pragma unroll
    for (int c8 = 0; c8 < DPT / 8; ++c8) {
      const float4 q0 = *reinterpret_cast<const float4*>(q + DPT * tig + 8 * c8), q1 = *reinterpret_cast<const float4*>(q + DPT * tig + 8 * c8 + 4);
      float kf[8];
      unpack8(*reinterpret_cast<const uint4*>(kx + DPT * tig + 8 * c8), kf);
      part += q0.x * kf[0] + q0.y * kf[1] + q0.z * kf[2] + q0.w * kf[3] + q1.x * kf[4] + q1.y * kf[5] + q1.z * kf[6] + q1.w * kf[7];
    }
    part += __shfl_xor_sync(0xffffffffu, part, 1);
    part += __shfl_xor_sync(0xffffffffu, part, 2);
    const float s_cur = part * qscale;
    const float M = fmaxf(m, s_cur);
    const float gs = ex2f(m - M);   // 0 when there is no history (m = -inf)
    const float pc = ex2f(s_cur - M);
    l = l * gs + pc;
#pragma unroll
    for (int nt = 0; nt < ND; ++nt) {
      const __nv_bfloat162 v2 = *reinterpret_cast<const __nv_bfloat162*>(vx + 8 * nt + 2 * tig);
      acc[nt][0] = fmaf(pc, __low2float(v2), acc[nt][0] * gs);
      acc[nt][1] = fmaf(pc, __high2float(v2), acc[nt][1] * gs);
    }
  }
  const float inv = __fdividef(1.f, l);
#pragma unroll
  for (int nt = 0; nt < ND; ++nt) { o[2 * nt] = acc[nt][0] * inv; o[2 * nt + 1] = acc[nt][1] * inv; }
}

__device__ __forceinline__ float4 ldg4(const float* p) { return __ldg(reinterpret_cast<const float4*>(p)); }

// DecodingManager.sift on one row, by one converged warp (postprocessing/postprocessing.py): softmax (:216),
// MemoryNode._look_back black list (:327-391), constrained arg-max (first maximum, like torch.argmax), MemoryNode.record
// (:303-325).  The masked probabilities are what the reference appends to its output (EfficientSATRN.py:553-555).
// Kept out of line: only rule-constrained decodes pay for its registers.
__device__ __noinline__ int sift_pick(const float* lrow, int V, int4* state, const int* __restrict__ flags, const int* __restrict__ limit,
                                      SiftIds ids, float* prow) {
  const int lane = threadIdx.x & 31;
  const int4 stt = *state;
  float mx = -INFINITY;
  for (int i = lane; i < V; i += 32) mx = fmaxf(mx, lrow[i]);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  float sum = 0.f;
  for (int i = lane; i < V; i += 32) sum += expf(lrow[i] - mx);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
  const int cur = stt.x;
  const int cf = (cur >= 0 && cur < V) ? __ldg(flags + cur) : 0;
  const int clim = (cur >= 0 && cur < V) ? __ldg(limit + cur) : 0;
  float best = -INFINITY;
  int bi = 0x7fffffff;
  for (int i = lane; i < V; i += 32) {
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
    const float pv = black ? 0.f : expf(lrow[i] - mx) / sum;
    if (prow) prow[i] = pv;
    if (pv > best) { best = pv; bi = i; }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float ob = __shfl_xor_sync(0xffffffffu, best, o);
    const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
    if (ob > best || (ob == best && oi < bi)) { best = ob; bi = oi; }
  }
  if (bi < 0 || bi >= V) bi = 0;
  __syncwarp();
  if (lane == 0) {
    int4 n = stt;
    n.y = (bi == stt.x) ? stt.y + 1 : 1;
    if (bi == ids.lbrace) n.z += 1;
    else if (bi == ids.rbrace) n.w += 1;
    n.x = bi;
    *state = n;
  }
  __syncwarp();
  return bi;
}
// Eight consecutive bias values of an epilogue unit, requested BEFORE the GEMM whose epilogue adds them (an L2 round
// trip inside the epilogue sat on the critical path of every one of the 19 stages of a step).
struct Bias8 { float4 a, b; };
__device__ __forceinline__ Bias8 ldg_bias8(const float* p, bool active) {
  Bias8 o;
  o.a = o.b = make_float4(0.f, 0.f, 0.f, 0.f);
  if (active) { o.a = ldg4(p); o.b = ldg4(p + 4); }
  return o;
}

}  // namespace

// ===========================================================================
// The persistent decode kernel
// ===========================================================================
#ifndef FRX_DEC_MINBLOCKS
#define FRX_DEC_MINBLOCKS (NTHR <= 256 ? 2 : 1)
#endif
__global__ void __cluster_dims__(CL, 1, 1) __launch_bounds__(NTHR, FRX_DEC_MINBLOCKS)
FRX_DEC_NAME(dec_cluster_bf16_kernel)(const DecClusterP p) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  Smem& s = *reinterpret_cast<Smem*>(smem_raw);
  EosRows& er = *reinterpret_cast<EosRows*>(smem_raw + sizeof(Smem));   // stop-at-<EOS> instantiations only
  cg::cluster_group cl = cg::this_cluster();
  const int r = (int)cl.block_rank();                        // CTA rank = head index = column slice
  const int img0 = p.img_base + (blockIdx.x / CL) * NIMG;    // first image of this cluster
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const uint64_t pol = make_evict_last_policy();
  const float qscale = 1.4426950408889634f / sqrtf((float)D);  // scores / sqrt(d_model), in exp2 units (see attend_mma)
  const float emb_scale = sqrtf((float)D);
  const int L = p.L, T = p.T, V = p.V, B = p.B;
  constexpr int LDA = D + APAD, LDA2 = FF + APAD;
  constexpr int KPD = D / 32, KPF = FF / 32;
  constexpr size_t WT = (size_t)KPD * 32;   // uint4 per tile for K = D
  constexpr int KS = 2;                     // every stage splits K over two warps
  // weight fragments (uint4 per lane) requested before the wait that precedes a stage
  constexpr int PF_A = GC<NTA, KPD, KS>::TOT > 16 ? GC<NTA, KPD, KS>::TPW : (GC<NTA, KPD, KS>::TOT < 6 ? GC<NTA, KPD, KS>::TOT : 6);
  constexpr int PF_S = GC<NTS, KPD, KS>::TOT;
  constexpr int PF_E = GC<NTE, KPD, KS>::TOT < 8 ? GC<NTE, KPD, KS>::TOT : 8;
  constexpr int PF_F = GC<NTS, KPF, KS>::TOT < 8 ? GC<NTS, KPF, KS>::TOT : 8;

  if (tid == 0) {
#pragma unroll
    for (int l = 0; l < 4; ++l) s.lw[l] = p.layer[l];
  }
  // ---- first input: <SOS> at position 0, or (step mode) the given token at the image's current position -----------
  for (int i = tid; i < NIMG * D; i += NTHR) {
    const int row = i / D, c = i % D;
    const int b = min(img0 + row, p.B - 1);
    long long tok = p.sos;
    if (p.first_tok32) tok = __ldg(p.first_tok32 + b);
    else if (p.first_tok64) tok = __ldg(p.first_tok64 + b);
    const int pos0 = p.hist_len ? __ldg(p.hist_len + b) : 0;
    float v = __ldg(p.emb + (size_t)tok * D + c) * emb_scale + __ldg(p.pe + (size_t)pos0 * D + c);
    s.xres[row][c] = v;
    s.abf[row][c] = __float2bfloat16_rn(v);
  }
  if (tid < NIMG) s.sift[tid] = make_int4(p.sift_ids.sos, 1, 0, 0);   // MemoryNode.__init__: <SOS>, run length 1, no braces
  const uint32_t bar0 = smem_u32(&s.bar[0]), bar1 = smem_u32(&s.bar[1]);
  if (tid == 0) {
    mbar_init(bar0, 1);
    mbar_init(bar1, 1);
    asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
  }
  // K/V ring: one mbarrier per (warp, slot), armed by the warp's lane 0 with every bulk request; the staging blocks start
  // as zeros so that rows a partial block never fills hold finite values (their probabilities are 0)
  if (KV_BULK) {
    if (lane == 0) {
#pragma unroll
      for (int d = 0; d < KVD; ++d) mbar_init(smem_u32(&s.kvbar[warp][d]), 1);
    }
    for (int i = tid; i < (int)(sizeof(s.kvst) / 16); i += NTHR) reinterpret_cast<uint4*>(&s.kvst[0][0][0][0][0])[i] = make_uint4(0u, 0u, 0u, 0u);
    asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");   // the zeros (generic proxy) precede the first bulk copy (async proxy)
  }
  __syncthreads();
  cl.sync();  // every CTA of the cluster is resident and its barriers initialised before the first remote store
  // Stage protocol: thread 0 arms the stage's barrier with the bytes THIS CTA will receive, everybody
  // computes and st.async-stores into all 8 CTAs, everybody waits for the local barrier phase.  A CTA can
  // run at most one exchange ahead of its slowest peer, and consecutive exchanges never share a buffer.
  int gstage = 0;
  auto stage_bar = [&]() -> uint32_t { return (gstage & 1) ? bar1 : bar0; };
  auto stage_begin = [&](uint32_t bytes) { if (tid == 0) mbar_expect_tx(stage_bar(), bytes); };
  auto stage_end = [&]() { mbar_wait(stage_bar(), (uint32_t)((gstage >> 1) & 1)); ++gstage; };
  int rsel = 0;
  auto next_red = [&]() -> float* { rsel ^= 1; return s.red[rsel]; };
  float* const logit_s = reinterpret_cast<float*>(&s.abf2[0][0]);  // [NIMG][LGS] fp32 view (abf2 is idle then)
  constexpr int LGS = VP + FPAD;
  static_assert(NIMG * LGS * 4 <= NIMG * (FF + APAD) * 2, "the fp32 logits view must fit in abf2");

  const bool profiling = p.prof != nullptr && blockIdx.x == 0 && tid == 0;
  if (profiling) for (int i = 0; i < 16; ++i) s.prof[i] = 0;
  long long tprev = clock64();
  auto mark = [&](int id) {
    if (profiling) {
      long long now = clock64();
      s.prof[id] += now - tprev;
      tprev = now;
    }
  };
  const int wimg = warp % NIMG, whc = warp / NIMG;  // this warp attends for image wimg, head r * HPC + whc
  const int head = r * HPC + whc;
  int b_mine = img0 + wimg;     // stop-at-<EOS>: the row's current image (-1: idle), re-read every step
  bool mine = b_mine < B;
  const int hist0 = (mine && p.hist_len) ? __ldg(p.hist_len + b_mine) : 0;      // keys cached before this launch
  const int* const chain = (mine && p.chain) ? p.chain + (size_t)b_mine * T : nullptr;
  KVStage* const kvst = reinterpret_cast<KVStage*>(&s.kvst[warp][0][0][0][0]);  // this warp's ring of K/V staging blocks
  const uint32_t kvbar = smem_u32(&s.kvbar[warp][0]);
  uint32_t kvphase = 0;   // bit d: parity of the next completion of ring slot d
  // Self K/V caches: [L][B][H][T][HD] by image, or (stop-at-<EOS>) [L][NSL][H][T][HD] by slot = cluster * 8 + row over all
  // of the launch's slots: any cluster may claim any image, so every slot may decode.  The grid has at most ceil(B / 8)
  // clusters, and the 16-bit self caches are allocated for max_batch rounded up to a multiple of 8.
  const int NSL = EOS ? (int)(gridDim.x / CL) * NIMG : B;
  const int kslot = EOS ? img0 + wimg : b_mine;   // cache slot of this warp's row

  // Stop-at-<EOS>: rows whose bit is set in `mask` take the next images from the work counter.  Every CTA of the cluster
  // takes the same decisions (the picks run on the gathered logits), so only the claimed index travels: rank 0 claims
  // one image per row and sends the first index on the stage mbarrier -- an exchange on steps where a row finished only.
  // Every CTA sends its word to every CTA (the others a dummy), so that, as for every other exchange, a CTA's wait ends
  // only when all its peers have reached the exchange: with rank 0 alone sending, a CTA could run two exchanges ahead of
  // a peer still waiting for the logits and complete that peer's barrier phase with the next step's stores.
  // Refilled rows restart at <SOS>, position 0, with a fresh MemoryNode state.
  auto refill = [&](uint32_t mask) {
    stage_begin(4u * CL);
    if (tid == 0) {
      const int first = r == 0 ? atomicAdd(p.work, __popc(mask)) : 0;
      for (int d = 0; d < CL; ++d) st_async_b32(mapa_u32(smem_u32(&er.claim[r]), d), (uint32_t)first, mapa_u32(stage_bar(), d));
    }
    stage_end();
    if (tid < NIMG && ((mask >> tid) & 1u)) {
      const int img = er.claim[0] + __popc(mask & ((1u << tid) - 1u));
      er.img[tid] = img < B ? img : -1;
      er.left[tid] = er.pos[tid] + 1;
      er.pos[tid] = 0;
      s.sift[tid] = make_int4(p.sift_ids.sos, 1, 0, 0);
    }
    for (int i = tid; i < NIMG * D; i += NTHR) {
      const int row = i / D, c = i % D;
      if (!((mask >> row) & 1u)) continue;
      const float v = __ldg(p.emb + (size_t)p.sos * D + c) * emb_scale + __ldg(p.pe + c);
      s.xres[row][c] = v;
      s.abf[row][c] = __float2bfloat16_rn(v);
    }
  };

  // all-gather of this warp's attention output (head r, image `warp`) into every CTA's obf: the eight gid
  // groups of the warp hold identical copies, group g serves destination CTA g
  auto store_attn = [&](uint32_t sb, const float (&o)[HD / 4]) {
    const uint32_t dst = (uint32_t)(lane >> 2);
    if (dst < (uint32_t)CL) {
      const uint32_t rb = mapa_u32(sb, dst);
      const uint32_t la = mapa_u32(smem_u32(&s.obf[wimg][head * HD + 2 * (lane & 3)]), dst);
#pragma unroll
      for (int nt = 0; nt < HD / 8; ++nt) st_async_b32(la + nt * 16, pack_bf16(o[2 * nt], o[2 * nt + 1]), rb);
    }
  };
  // epilogue of a "pre-LayerNorm" stage: 8 columns of row `row`, + bias (+ ReLU) + residual, sent to CTA `sub`
  // (bias: the unit's 8 values, loaded by pre_bias() before the stage)
  auto pre_bias = [&](const float* bias) {   // unit of this thread in an NTS-tile stage: tile = (tid % (NTS * 8)) >> 3
    return ldg_bias8(bias + r * SW + ((tid % (NTS * 8)) >> 3) * 8, true);
  };
  auto pre_epi = [&](uint32_t sb, const Bias8& bias, bool relu) {
    return [&, sb, bias, relu](int tile, int row, float (&v)[8], int sub) {
      // NSUB threads share a unit and split the CL destination CTAs between them (one each when NSUB >= CL)
      constexpr int NSUB_S = GC<NTS, KPD, KS>::NSUB, DPT = (CL + NSUB_S - 1) / NSUB_S;
      if (sub * DPT >= CL) return;
      const int col = r * SW + tile * 8;
      const float4 b0 = bias.a, b1 = bias.b;
      const float4 x0 = *reinterpret_cast<const float4*>(&s.xres[row][col]), x1 = *reinterpret_cast<const float4*>(&s.xres[row][col + 4]);
      float o[8] = {v[0] + b0.x, v[1] + b0.y, v[2] + b0.z, v[3] + b0.w, v[4] + b1.x, v[5] + b1.y, v[6] + b1.z, v[7] + b1.w};
      if (relu) {
#pragma unroll
        for (int i = 0; i < 8; ++i) o[i] = fmaxf(o[i], 0.f);
      }
      const uint4 lo = make_uint4(__float_as_uint(o[0] + x0.x), __float_as_uint(o[1] + x0.y), __float_as_uint(o[2] + x0.z), __float_as_uint(o[3] + x0.w));
      const uint4 hi = make_uint4(__float_as_uint(o[4] + x1.x), __float_as_uint(o[5] + x1.y), __float_as_uint(o[6] + x1.z), __float_as_uint(o[7] + x1.w));
#pragma unroll
      for (int d = 0; d < DPT; ++d) {
        const uint32_t dst = (uint32_t)(sub * DPT + d);
        if (dst >= (uint32_t)CL) break;
        const uint32_t la = mapa_u32(smem_u32(&s.pre[row][col]), dst), rb = mapa_u32(sb, dst);
        st_async_v4(la, lo, rb);
        st_async_v4(la + 16, hi, rb);
      }
    };
  };
  // q|k|v of head r (tiles: q 0-3, k 4-7, v 8-11), biases at `bias` in natural [q|k|v] column order
  auto qkv_bias = [&](const float* bias) {   // this thread's unit in the NTA-tile stage (sub 0 only: tid < NTA * 8)
    const int tile = tid >> 3, seg = tile / NTS, wc = (tile % NTS) * 8;
    return ldg_bias8(bias + seg * D + r * SW + wc, tid < NTA * 8);
  };
  auto qkv_epi = [&](const Bias8& bias) {
    return [&, bias](int tile, int row, float (&v)[8], int sub) {
      if (sub != 0) return;
      const int seg = tile / NTS, wc = (tile % NTS) * 8, hc = wc / HD, col = wc % HD;  // column wc of this CTA's slice
      const float4 b0 = bias.a, b1 = bias.b;
      const float o[8] = {v[0] + b0.x, v[1] + b0.y, v[2] + b0.z, v[3] + b0.w, v[4] + b1.x, v[5] + b1.y, v[6] + b1.z, v[7] + b1.w};
      if (seg == 0) {
        *reinterpret_cast<float4*>(&s.qh[hc][row][col]) = make_float4(o[0], o[1], o[2], o[3]);
        *reinterpret_cast<float4*>(&s.qh[hc][row][col + 4]) = make_float4(o[4], o[5], o[6], o[7]);
      } else {
        __nv_bfloat16(*dst)[HD + APAD] = seg == 1 ? s.kcur[hc] : s.vcur[hc];
        *reinterpret_cast<uint4*>(&dst[row][col]) =
            make_uint4(pack_bf16(o[0], o[1]), pack_bf16(o[2], o[3]), pack_bf16(o[4], o[5]), pack_bf16(o[6], o[7]));
      }
    };
  };
  // K/V cache rows (layer lc, position t) of the rows in abf: tiles 0-3 = K of head r, 4-7 = V of head r
  auto cache_rows = [&](int lc, int t, const uint4* wp, const float* bias) {
    const Bias8 cb = ldg_bias8(bias + ((tid >> 3) / NTS) * D + r * SW + ((tid >> 3) % NTS) * 8, tid < NTC * 8);
    gemm2<NTC, KPD, KS>(next_red(), &s.abf[0][0], LDA, wp, pol, WPre<0>{}, [&](int tile, int row, float (&v)[8], int sub) {
      const int b = img0 + row;   // stop-at-<EOS>: the row's slot
      if (sub != 0 || (EOS ? er.img[row] < 0 : b >= B)) return;
      const int seg = tile / NTS, wc = (tile % NTS) * 8, hd = r * HPC + wc / HD, col = wc % HD;
      const float4 b0 = cb.a, b1 = cb.b;
      __nv_bfloat16* dst = seg == 0 ? p.kself : p.vself;
      const int wrow = EOS ? er.pos[row]
                           : (p.slot ? __ldg(p.slot + b) : (p.hist_len ? __ldg(p.hist_len + b) : 0)) + t;   // cache row of this step
      *reinterpret_cast<uint4*>(dst + (((((size_t)lc * NSL + b) * H + hd) * T) + wrow) * HD + (((col >> 3) ^ kv_perm(wrow)) << 3)) =
          make_uint4(pack_bf16(v[0] + b0.x, v[1] + b0.y), pack_bf16(v[2] + b0.z, v[3] + b0.w),
                     pack_bf16(v[4] + b1.x, v[5] + b1.y), pack_bf16(v[6] + b1.z, v[7] + b1.w));
      // the row is read back by bulk copies (async proxy) from the next step on: order this generic-proxy write before them
      if (KV_BULK) asm volatile("fence.proxy.async.global;\n" ::: "memory");
    });
  };

  auto pre_a = prefetch_w<NTA, KPD, KS, PF_A>(p.w_first + (size_t)r * NTA * WT, pol);
  // The K/V ring is idle between two attention phases, so the first blocks of the NEXT phase are requested as soon as
  // the current one has handed its result over: the cross K/V of a layer right after its self-attention, the self K/V of
  // the next layer (next step: layer 0, whose newest cache row was written during this step's layer 1) right after the
  // cross-attention -- they land under the stages in between instead of under one short projection.
  auto prime_self = [&](int l, int t) {
    const size_t base = ((((size_t)l * NSL + (mine ? kslot : 0)) * H + head) * T) * HD;
    kv_prime(kvst, p.kself + base, p.vself + base, mine ? hist0 + t : 0, chain, kvbar);
  };
  auto prime_cross = [&](int l) {
    const size_t base = ((((size_t)l * B + (mine ? b_mine : 0)) * H + head) * p.S) * HD;
    kv_prime(kvst, p.kcross + base, p.vcross + base, mine ? p.S : 0, nullptr, kvbar);
  };
  if constexpr (EOS) {   // every row starts with a claimed image
    if (tid < NIMG) { er.pos[tid] = 0; er.done[tid] = 0; }
    refill(0xffu);
    __syncthreads();
    b_mine = er.img[wimg];
    mine = b_mine >= 0;
  }
  prime_self(0, 0);
  bool self_primed = true;
  for (int t = 0; EOS || t < p.steps; ++t) {
    // position of this warp's row, re-read where it is used (a register for it through the step would spill)
    const auto tpos = [&]() { return EOS ? er.pos[wimg] : t; };
    if constexpr (EOS) {
      b_mine = er.img[wimg];
      mine = b_mine >= 0;
    }
    for (int l = 0; l < L; ++l) {
      const DecClusterLayer& W = s.lw[l];
      // ---- A: q|k|v of head r from the layer input, then self attention of (image warp, head r) -------
      {
        const size_t base = ((((size_t)l * NSL + (mine ? kslot : 0)) * H + head) * T) * HD;
        const int n_hist = mine ? hist0 + tpos() : 0;
        if constexpr (EOS && EARLY_PRIME) {
          // the blocks requested for this step at the end of the last one belong to a history the row has left (it
          // finished, was refilled or went idle): let them land, then request the row's own
          if (l == 0 && self_primed && er.done[wimg]) {
            const int primed_n = er.left[wimg];   // what the last step's early prime requested (mine: the row was busy)
#pragma unroll
            for (int d = 0; d < KVD; ++d) {
              if (32 * d < primed_n) {
                mbar_wait(kvbar + 8u * d, (kvphase >> d) & 1u);
                kvphase ^= 1u << d;
              }
            }
            __syncwarp();
            self_primed = false;
          }
        }
        if (!self_primed) prime_self(l, tpos());   // single-layer decoders only: the newest cache row is written late in the step
        self_primed = false;
        const uint4* wp = l == 0 ? p.w_first + (size_t)r * NTA * WT : s.lw[l - 1].w_next + ((size_t)r * (NTC + NTA) + NTC) * WT;
        const Bias8 bias = qkv_bias(l == 0 ? p.b_first : s.lw[l - 1].b_next + 2 * D);
        gemm2<NTA, KPD, KS>(next_red(), &s.abf[0][0], LDA, wp, pol, pre_a, qkv_epi(bias));
        __syncthreads();
        mark(0);
        stage_begin(NIMG * D * 2u);
        const uint32_t sb = stage_bar();
        float o[HD / 4];
        if (!KV_BULK || chain)
          attend_mma<false>(kvst, &s.qh[whc][wimg][0], p.kself + base, p.vself + base, n_hist, chain, kvbar, kvphase, &s.kcur[whc][wimg][0], &s.vcur[whc][wimg][0], qscale, o,
                            profiling ? &s.prof[11] : nullptr);
        else
          attend_mma<true>(kvst, &s.qh[whc][wimg][0], p.kself + base, p.vself + base, n_hist, nullptr, kvbar, kvphase, &s.kcur[whc][wimg][0], &s.vcur[whc][wimg][0], qscale, o,
                           profiling ? &s.prof[11] : nullptr);
        store_attn(sb, o);
        if (EARLY_PRIME) prime_cross(l);
        mark(1);
      }
      const auto pre_b = prefetch_w<NTS, KPD, KS, PF_S>(W.w_o + (size_t)r * NTS * WT, pol);
      const Bias8 bias_b = pre_bias(W.b_o);
      // nobody waits for this in the current step: cache rows of the previous layer's output (= this input)
      if (l > 0) cache_rows(l - 1, t, s.lw[l - 1].w_next + (size_t)r * (NTC + NTA) * WT, s.lw[l - 1].b_next);
      mark(2);
      stage_end();
      mark(3);
      // ---- B: out_linear(a) + x -> pre ; LN -> u -----------------------------------------
      stage_begin(NIMG * D * 4u);
      gemm2<NTS, KPD, KS>(next_red(), &s.obf[0][0], LDA, W.w_o + (size_t)r * NTS * WT, pol, pre_b, pre_epi(stage_bar(), bias_b, false));
      mark(4);
      const LnParams lnp1 = load_ln(W.ln1_g, W.ln1_b);
      const auto pre_c = prefetch_w<NTS, KPD, KS, PF_S>(W.w_q2 + (size_t)r * NTS * WT, pol);
      const Bias8 bias_c = ldg_bias8(W.b_q2 + r * SW + (tid >> 3) * 8, tid < NTS * 8);
      stage_end();
      mark(5);
      layernorm_rows(s, lnp1);
      __syncthreads();
      mark(6);
      // ---- C: q2 of head r, cross attention of (image warp, head r) over the S memory tokens -------
      {
        const size_t base = ((((size_t)l * B + (mine ? b_mine : 0)) * H + head) * p.S) * HD;
        const int n_keys = mine ? p.S : 0;
        if (!EARLY_PRIME) prime_cross(l);
        gemm2<NTS, KPD, KS>(next_red(), &s.abf[0][0], LDA, W.w_q2 + (size_t)r * NTS * WT, pol, pre_c,
                          [&](int tile, int row, float (&v)[8], int sub) {
                            if (sub != 0) return;
                            const int wc = tile * 8, hc = wc / HD, col = wc % HD;
                            const float4 b0 = bias_c.a, b1 = bias_c.b;
                            *reinterpret_cast<float4*>(&s.qh[hc][row][col]) = make_float4(v[0] + b0.x, v[1] + b0.y, v[2] + b0.z, v[3] + b0.w);
                            *reinterpret_cast<float4*>(&s.qh[hc][row][col + 4]) = make_float4(v[4] + b1.x, v[5] + b1.y, v[6] + b1.z, v[7] + b1.w);
                          });
        __syncthreads();
        mark(4);
        stage_begin(NIMG * D * 2u);
        const uint32_t sb = stage_bar();
        float o[HD / 4];
        if (mine) {
          attend_mma<KV_BULK>(kvst, &s.qh[whc][wimg][0], p.kcross + base, p.vcross + base, n_keys, nullptr, kvbar, kvphase, nullptr, nullptr, qscale, o);
        } else {
#pragma unroll
          for (int i = 0; i < HD / 4; ++i) o[i] = 0.f;
        }
        store_attn(sb, o);
        if (EARLY_PRIME) {
          if (l + 1 < L) { prime_self(l + 1, tpos()); self_primed = true; }
          else if (L >= 2 && (EOS || t + 1 < p.steps)) {
            prime_self(0, tpos() + 1);
            self_primed = true;
          }
        }
        mark(7);
      }
      const auto pre_d = prefetch_w<NTS, KPD, KS, PF_S>(W.w_o2 + (size_t)r * NTS * WT, pol);
      const Bias8 bias_d = pre_bias(W.b_o2);
      stage_end();
      mark(3);
      // ---- D: out_linear(c) + u -> pre ; LN -> w ------------------------------------------------
      stage_begin(NIMG * D * 4u);
      gemm2<NTS, KPD, KS>(next_red(), &s.obf[0][0], LDA, W.w_o2 + (size_t)r * NTS * WT, pol, pre_d, pre_epi(stage_bar(), bias_d, false));
      mark(4);
      const LnParams lnp2 = load_ln(W.ln2_g, W.ln2_b);
      const auto pre_e = prefetch_w<NTE, KPD, KS, PF_E>(W.w_f0 + (size_t)r * NTE * WT, pol);
      const Bias8 bias_e = ldg_bias8(W.b_f0 + r * FS + ((tid % (NTE * 8)) >> 3) * 8, true);
      stage_end();
      mark(5);
      layernorm_rows(s, lnp2);
      __syncthreads();
      mark(6);
      // ---- E: ff = relu(linear0(w)); CTA r owns hidden units [128r, 128r+128) ------------------------
      {
        stage_begin(NIMG * FF * 2u);
        const uint32_t sb = stage_bar();
        gemm2<NTE, KPD, KS>(next_red(), &s.abf[0][0], LDA, W.w_f0 + (size_t)r * NTE * WT, pol, pre_e,
                           [&](int tile, int row, float (&v)[8], int sub) {
                             const int col = r * FS + tile * 8;
                             const float4 b0 = bias_e.a, b1 = bias_e.b;
                             const uint4 o = make_uint4(pack_bf16(fmaxf(v[0] + b0.x, 0.f), fmaxf(v[1] + b0.y, 0.f)),
                                                        pack_bf16(fmaxf(v[2] + b0.z, 0.f), fmaxf(v[3] + b0.w, 0.f)),
                                                        pack_bf16(fmaxf(v[4] + b1.x, 0.f), fmaxf(v[5] + b1.y, 0.f)),
                                                        pack_bf16(fmaxf(v[6] + b1.z, 0.f), fmaxf(v[7] + b1.w, 0.f)));
                             const uint32_t la = smem_u32(&s.abf2[row][col]);
                             constexpr int NSUB_E = GC<NTE, KPD, KS>::NSUB, DPT = (CL + NSUB_E - 1) / NSUB_E;  // destinations per thread
#pragma unroll
                             for (int d = 0; d < DPT; ++d) {
                               const uint32_t dst = (uint32_t)(sub * DPT + d);
                               if (dst < (uint32_t)CL) st_async_v4(mapa_u32(la, dst), o, mapa_u32(sb, dst));
                             }
                           });
        mark(8);
      }
      const auto pre_f = prefetch_w<NTS, KPF, KS, PF_F>(W.w_f1 + (size_t)r * NTS * KPF * 32, pol);
      const Bias8 bias_f = pre_bias(W.b_f1);
      stage_end();
      mark(5);
      // ---- F: relu(linear1(ff)) + w -> pre ; LN -> y -----------------------------------------------
      stage_begin(NIMG * D * 4u);
      gemm2<NTS, KPF, KS>(next_red(), &s.abf2[0][0], LDA2, W.w_f1 + (size_t)r * NTS * KPF * 32, pol, pre_f, pre_epi(stage_bar(), bias_f, true));
      mark(9);
      const LnParams lnp3 = load_ln(W.ln3_g, W.ln3_b);
      const bool last_layer = l + 1 >= L;
      // next consumer of y: the next layer's q|k|v (12 tiles), or the generator (4 tiles); both sit behind
      // the 8 cache tiles in w_next
      constexpr int PF_G = GC<NG, KPD, KS>::TOT;
      WPre<PF_G> pre_g;
      float gbias[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) gbias[i] = 0.f;
      if (!last_layer) pre_a = prefetch_w<NTA, KPD, KS, PF_A>(W.w_next + ((size_t)r * (NTC + NTA) + NTC) * WT, pol);
      else {
        pre_g = prefetch_w<NG, KPD, KS, PF_G>(W.w_next + ((size_t)r * (NTC + NG) + NTC) * WT, pol);
        const int col = r * (VP / CL) + ((tid % (NG * 8)) >> 3) * 8;
        const float* gb = W.b_next + 2 * D;
        if (tid < NG * 8 * CL) {
#pragma unroll
          for (int i = 0; i < 8; ++i) gbias[i] = col + i < V ? __ldg(gb + col + i) : 0.f;
        }
      }
      stage_end();
      mark(5);
      layernorm_rows(s, lnp3);
      __syncthreads();
      mark(6);
      if (last_layer) {
        // ---- G: vocabulary logits (V columns padded to 256; CTA r owns [32r, 32r+32)) ------------------
        stage_begin(NIMG * VP * 4u);
        const uint32_t sb = stage_bar();
        gemm2<NG, KPD, KS>(next_red(), &s.abf[0][0], LDA, W.w_next + ((size_t)r * (NTC + NG) + NTC) * WT, pol, pre_g,
                          [&](int tile, int row, float (&v)[8], int sub) {
                            constexpr int NSUB_G = GC<NG, KPD, KS>::NSUB, DPT = (CL + NSUB_G - 1) / NSUB_G;
                            if (sub * DPT >= CL) return;
                            const int col = r * (VP / CL) + tile * 8;
#pragma unroll
                            for (int i = 0; i < 8; ++i) v[i] += gbias[i];
#pragma unroll
                            for (int d = 0; d < DPT; ++d) {
                              const uint32_t dst = (uint32_t)(sub * DPT + d);
                              if (dst >= (uint32_t)CL) break;
                              const uint32_t la = mapa_u32(smem_u32(logit_s + row * LGS + col), dst), rb = mapa_u32(sb, dst);
                              st_async_v4(la, make_uint4(__float_as_uint(v[0]), __float_as_uint(v[1]), __float_as_uint(v[2]), __float_as_uint(v[3])), rb);
                              st_async_v4(la + 16, make_uint4(__float_as_uint(v[4]), __float_as_uint(v[5]), __float_as_uint(v[6]), __float_as_uint(v[7])), rb);
                            }
                            const int b = EOS ? er.img[row] : img0 + row;
                            if (sub == (CL > 1 ? 1 : 0) && p.logits && (EOS ? b >= 0 : b < B) && !p.sift_flags) {
                              float* lp = p.logits + ((size_t)b * p.steps + (EOS ? er.pos[row] : t)) * V + col;
#pragma unroll
                              for (int i = 0; i < 8; ++i)
                                if (col + i < V) lp[i] = v[i];
                            }
                          });
        mark(4);
        pre_a = prefetch_w<NTA, KPD, KS, PF_A>(p.w_first + (size_t)r * NTA * WT, pol);
        cache_rows(l, t, W.w_next + (size_t)r * (NTC + NG) * WT, W.b_next);
        mark(2);
        stage_end();
        mark(5);
      }
    }  // layers
    // ---- greedy pick (first max index) + next input: warp w <-> row w, every CTA does all rows ----------
    if (warp < NIMG) {
      const int row = warp;
      int bi;
      if (p.sift_flags) {
        float* prow = (mine && r == 0 && p.logits) ? p.logits + ((size_t)b_mine * p.steps + tpos()) * V : nullptr;
        bi = sift_pick(logit_s + row * LGS, V, &s.sift[row], p.sift_flags, p.sift_limit, p.sift_ids, prow);
      } else {
        float best = -INFINITY;
        bi = 0x7fffffff;
        for (int i = lane; i < V; i += 32) {
          float v = logit_s[row * LGS + i];
          if (v > best) { best = v; bi = i; }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
          float ob = __shfl_xor_sync(0xffffffffu, best, o);
          int oi = __shfl_xor_sync(0xffffffffu, bi, o);
          if (ob > best || (ob == best && oi < bi)) { best = ob; bi = oi; }
        }
        if (bi < 0 || bi >= V) bi = 0;
      }
      int nxt = bi;
      if (mine) {
        if (p.forced) nxt = (int)p.forced[(size_t)b_mine * p.steps + tpos()];
        if (r == 0 && lane == 0 && p.tokens) p.tokens[(size_t)b_mine * p.steps + tpos()] = bi;
      }
      bool more = t + 1 < p.steps;
      if constexpr (EOS) {   // the row stops after the step that emits (forced: is fed) <EOS>, or after the last step
        more = mine && nxt != p.eos && tpos() + 1 < p.steps;
        if (mine && !more && r == 0 && lane == 0) p.lengths[b_mine] = tpos() + 1;
        if (lane == 0) er.done[row] = mine && !more;
      }
      if (more) {
        const float* pe = p.pe + (size_t)(hist0 + tpos() + 1) * D;
#pragma unroll
        for (int i = 0; i < D / 32; ++i) {
          const int c = i * 32 + lane;
          float v = __ldg(p.emb + (size_t)nxt * D + c) * emb_scale + __ldg(pe + c);
          s.xres[row][c] = v;
          s.abf[row][c] = __float2bfloat16_rn(v);
        }
      }
    }
    __syncthreads();
    mark(10);
    if constexpr (EOS) {
      uint32_t finished = 0;
#pragma unroll
      for (int i = 0; i < NIMG; ++i) finished |= (er.done[i] ? 1u : 0u) << i;
      if (tid < NIMG && er.img[tid] >= 0 && !((finished >> tid) & 1u)) er.pos[tid] += 1;
      if (finished) refill(finished);
      __syncthreads();
      bool busy = false;
#pragma unroll
      for (int i = 0; i < NIMG; ++i) busy = busy || er.img[i] >= 0;
      if (!busy) {   // the same decision in every CTA of the cluster
        if constexpr (EARLY_PRIME) {
          // a row that finished in this step has K/V blocks in flight, requested for a next step that will not come: they
          // must land before the CTA exits, or a bulk copy completes into the shared memory of the next CTA on this SM
          if (self_primed && er.done[wimg]) {
            const int primed_n = er.left[wimg];
#pragma unroll
            for (int d = 0; d < KVD; ++d) {
              if (32 * d < primed_n) {
                mbar_wait(kvbar + 8u * d, (kvphase >> d) & 1u);
                kvphase ^= 1u << d;
              }
            }
            __syncwarp();
          }
        }
        break;
      }
    }
  }
  cl.sync();  // nobody exits while a peer's stores to it may still be in flight
  if (profiling) for (int i = 0; i < 16; ++i) p.prof[i] = s.prof[i];
}

size_t FRX_DEC_NAME(dec_cluster_smem_bytes)() { return SMEM_BYTES; }

// One launch decodes up to DEC_MAX_CLUSTERS clusters (all co-resident: two CTAs per SM); larger batches
// are decoded in consecutive launches over image ranges.  The stop-at-<EOS> instantiations decode any batch in one
// launch of at most DEC_MAX_CLUSTERS clusters whose rows take images from the work counter.
int FRX_DEC_NAME(launch_dec_cluster_bf16)(const DecClusterP& p0, cudaStream_t st) {
  static SmemOptIn opt;
  {
    cudaError_t e = opt.ensure(FRX_DEC_NAME(dec_cluster_bf16_kernel), SMEM_BYTES, true);
    if (e != cudaSuccess) return (int)e;
  }
  if (EOS) {
    const int clusters = (p0.B + NIMG - 1) / NIMG < DEC_MAX_CLUSTERS ? (p0.B + NIMG - 1) / NIMG : DEC_MAX_CLUSTERS;
    FRX_DEC_NAME(dec_cluster_bf16_kernel)<<<clusters * CL, NTHR, SMEM_BYTES, st>>>(p0);
    return 0;
  }
  if (getenv("FRX_DEBUG")) {
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(DEC_MAX_CLUSTERS * CL); cfg.blockDim = dim3(NTHR); cfg.dynamicSmemBytes = SMEM_BYTES;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = CL; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.attrs = at; cfg.numAttrs = 1;
    int n = -1;
    cudaError_t e = cudaOccupancyMaxActiveClusters(&n, FRX_DEC_NAME(dec_cluster_bf16_kernel), &cfg);
    fprintf(stderr, "[frx] decode kernel: clusters of %d CTAs x %d threads, max co-resident clusters = %d (%s), smem %zu B\n",
            CL, NTHR, n, cudaGetErrorString(e), SMEM_BYTES);
  }
  for (int base = 0; base < p0.B; base += DEC_MAX_CLUSTERS * NIMG) {
    DecClusterP p = p0;
    p.img_base = base;
    const int n = p0.B - base < DEC_MAX_CLUSTERS * NIMG ? p0.B - base : DEC_MAX_CLUSTERS * NIMG;
    const int clusters = (n + NIMG - 1) / NIMG;
    FRX_DEC_NAME(dec_cluster_bf16_kernel)<<<clusters * CL, NTHR, SMEM_BYTES, st>>>(p);
  }
  return 0;
}

#ifndef FRX_DEC_VARIANT
// ===========================================================================
// cross K/V: fp32 [B*S][L*2*D] (k_l | v_l per layer) -> bf16 head-major
// [L][B][H][S][32] caches
// ===========================================================================
__global__ void __launch_bounds__(256) cross_to_bf16_kernel(const float* __restrict__ src, __nv_bfloat16* __restrict__ kc,
                                                            __nv_bfloat16* __restrict__ vc, int B, int S, int L, int Dm, int hd) {
  // one thread = 8 consecutive features of one head (32-byte load, 16-byte store)
  const int Hh = Dm / hd, cols8 = L * 2 * Dm / 8;
  long long total = (long long)B * S * cols8;
  long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= total) return;
  int col = (int)(idx % cols8) * 8;
  long long row = idx / cols8;
  int sidx = (int)(row % S), b = (int)(row / S);
  int l = col / (2 * Dm), which = (col / Dm) & 1, d = col % Dm;
  int hh = d / hd, dd = d % hd;
  // rows keep their 16-byte chunks in the permuted order the decode kernel's staging blocks use (kv_perm there)
  const int perm = hd == 32 ? ((sidx >> 1) & 3) : (sidx & (hd / 8 - 1));
  dd = ((dd >> 3) ^ perm) << 3;
  size_t off = (((((size_t)l * B + b) * Hh + hh) * S) + sidx) * hd + dd;
  const float4 a = __ldg(reinterpret_cast<const float4*>(src + idx * 8)), c = __ldg(reinterpret_cast<const float4*>(src + idx * 8) + 1);
  const __nv_bfloat162 p0 = __floats2bfloat162_rn(a.x, a.y), p1 = __floats2bfloat162_rn(a.z, a.w);
  const __nv_bfloat162 p2 = __floats2bfloat162_rn(c.x, c.y), p3 = __floats2bfloat162_rn(c.z, c.w);
  *reinterpret_cast<uint4*>((which ? vc : kc) + off) =
      make_uint4(*reinterpret_cast<const uint32_t*>(&p0), *reinterpret_cast<const uint32_t*>(&p1),
                 *reinterpret_cast<const uint32_t*>(&p2), *reinterpret_cast<const uint32_t*>(&p3));
}

void launch_cross_to_bf16(const float* src, __nv_bfloat16* kc, __nv_bfloat16* vc, int B, int S, int L, int Dm, int head_dim,
                          cudaStream_t st) {
  long long total = (long long)B * S * L * 2 * Dm / 8;
  cross_to_bf16_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(src, kc, vc, B, S, L, Dm, head_dim);
}

#endif  // FRX_DEC_VARIANT

}  // namespace frx
