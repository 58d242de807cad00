// kernels.h -- host-callable launchers of the frx kernels.
#pragma once
#include "common.cuh"

namespace frx {

// fp32 kernel set (kernels_f32.cu)
void launch_stem_conv(const float* in, const float* w, const float* scale, const float* shift, float* out,
                      int B, int Cin, int H, int W, int OH, int OW, int Cout, cudaStream_t st);
void launch_direct_conv3x3(const float* in, const float* w, const float* scale, const float* shift, float* out, int B,
                           int Cin, int H, int W, int OH, int OW, int Cout, int stride, int pad, int act,
                           cudaStream_t st);
void launch_igemm_f32(const GemmP& p, cudaStream_t st);
void launch_dwconv_f32(const DwP& p, cudaStream_t st);
void launch_se_gate_f32(const float* x, const float* w1, const float* b1, const float* w2, const float* b2,
                        float* gate, int B, int HW, int C, int R, cudaStream_t st);
void launch_maxpool2_f32(const float* in, float* out, int B, int H, int W, int C, cudaStream_t st);
void launch_pe2d_f32(const float* x, const float* w0, const float* b0, const float* w1, const float* b1,
                     const float* peh, const float* pew, float* out, int B, int h, int w, int C,
                     cudaStream_t st);
void launch_layernorm_f32(const float* x, const float* res, const float* gamma, const float* beta, float* out,
                          int M, int C, int scramble_S, cudaStream_t st);
void launch_enc_attn_f32(const float* qkv, float* out, int B, int S, int D, int heads, cudaStream_t st);
void launch_dec_gemm_f32(const DecGemmP& p, cudaStream_t st);
void launch_dec_attn_f32(const AttnP& p, int head_dim, cudaStream_t st);
// training-step variants with attention dropout on the probabilities (common.cuh DropP)
void launch_enc_attn_f32_drop(const float* qkv, float* out, int B, int S, int D, int heads, const DropP& drop, cudaStream_t st);
void launch_dec_attn_f32_drop(const AttnP& p, int head_dim, const DropP& drop, cudaStream_t st);
void launch_fill_i32(int* p, int v, int n, cudaStream_t st);
void launch_dec_embed_f32(const int* tok, const long long* tok64, int fixed_token, const float* emb,
                          const float* pe, int pos, const int* pos_arr, int pos_mod, float scale, float* x,
                          int M, int D, cudaStream_t st);
void launch_dec_argmax_embed(const float* logits, long long ld_logits, int V, long long* tokens_out,
                             long long ld_tok, const long long* forced, long long ld_forced, int* cur_tok,
                             const float* emb, const float* pe_next, float scale, float* x, int M, int D,
                             cudaStream_t st);


void launch_dec_sift_embed(float* logits, long long ld_logits, int V, long long* tokens_out, long long ld_tok, int4* state,
                           const int* flags, const int* limit, const SiftIds& ids, int* cur_tok, const float* emb,
                           const float* pe_next, float scale, float* x, int M, int D, cudaStream_t st);
void launch_sift_state_init(int4* state, int M, int sos, cudaStream_t st);
void launch_pad_mask(const long long* text, unsigned char* mask, int B, int L, int pad_id, cudaStream_t st);
void launch_eos_finalize(float* logits, long long* tokens, int* lengths, const long long* stop, int B, int steps, int V,
                         int eos, int pad, bool have_len, cudaStream_t st);

// SwinTRN encoder pieces (kernels_swin.cu)
void launch_swin_patch_embed(const float* img, const float* w, const float* bias, const float* g, const float* b,
                             const float* ape, float* out, int B, int IMGS, int R, int E, cudaStream_t st);
void launch_swin_window_attn(const float* qkv, const float* bias_table, float* out, int B, int R, int C, int heads, int ws,
                             int shift, cudaStream_t st);
bool launch_swin_window_attn_mma(const float* qkv, const float* bias_table, eh_t* out, int B, int R, int C, int heads,
                                 int ws, int shift, cudaStream_t st);
void launch_swin_patch_merge(const float* x, float* out, int B, int R, int C, cudaStream_t st);

// best-first search bookkeeping (kernels_beam.cu)
void launch_beam_init(const BeamP& p, cudaStream_t st);
void launch_beam_select(const BeamP& p, cudaStream_t st);
void launch_beam_push(const BeamP& p, cudaStream_t st);
void launch_beam_finish(const BeamP& p, cudaStream_t st);

// tcgen05 implicit GEMM + bf16 trunk kernels (kernels_tc.cu, kernels_bf16.cu)
int launch_tc_igemm(TcGemmP p, cudaStream_t st);                       // one tile per CTA (first version)
int launch_tc_igemm_ws(TcGemmP p, int num_sms, cudaStream_t st);       // persistent, warp-specialised
void launch_pad_conv_weights(const eh_t* in, eh_t* out, long long rows, int Cin, cudaStream_t st);
void launch_h16_to_f32(const eh_t* in, float* out, long long n, cudaStream_t st);
void launch_f32_to_h16(const float* in, eh_t* out, long long n, cudaStream_t st);
void launch_stem_conv_bf16(const float* in, const float* w, const float* scale, const float* shift,
                           eh_t* out, int B, int Cin, int H, int W, int OH, int OW, int Cout, cudaStream_t st);
void launch_dwconv_bf16(const eh_t* in, const float* w, const float* scale, const float* shift,
                        eh_t* out, int B, int H, int W, int C, int OH, int OW, int stride, int pad_t,
                        int pad_l, int act, cudaStream_t st);
void launch_se_scale_bf16(eh_t* x, const float* w1, const float* b1, const float* w2, const float* b2,
                          int B, int HW, int C, int R, cudaStream_t st);
void launch_mbconv_dw_se_bf16(const eh_t* in, const float* w, const float* scale, const float* shift,
                              eh_t* out, float* mean, float* gate, const float* w1, const float* b1,
                              const float* w2, const float* b2, int B, int H, int W, int C, int OH, int OW, int stride,
                              int pad_t, int pad_l, int R, cudaStream_t st);
void launch_layernorm_bf16out(const float* x, const float* res, const float* gamma, const float* beta,
                              eh_t* out, int M, int C, int scramble_S, cudaStream_t st);
void launch_enc_attn_bf16out(const float* qkv, eh_t* out, int B, int S, int D, int heads, cudaStream_t st);
void launch_conv3x3_c24_bf16(const eh_t* in, const void* wfrag, const float* scale, const float* shift,
                             eh_t* out, int B, int H, int W, int add_res, cudaStream_t st);
void launch_lite_conv0_pool_bf16(const float* in, const float* w, const float* scale, const float* shift, eh_t* out,
                                 int B, int Cin, int H, int W, int Cout, cudaStream_t st);
void launch_maxpool2_bf16(const eh_t* in, eh_t* out, float* out_f32, int B, int H, int W, int C, cudaStream_t st);
bool launch_enc_attn_mma_bf16(const float* qkv, eh_t* out, int B, int S, int D, int heads, cudaStream_t st);

// bf16 persistent decode (kernels_decode_bf16.cu)
size_t dec_cluster_smem_bytes();
int launch_dec_cluster_bf16(const DecClusterP& p, cudaStream_t st);       // hidden 256, 8 heads, filter 1024 (clusters of 8)
int launch_dec_cluster_bf16_d128(const DecClusterP& p, cudaStream_t st);  // hidden 128, 4 heads, filter 512 (clusters of 4)
int launch_dec_cluster_bf16_p2(const DecClusterP& p, cudaStream_t st);    // hidden 256, two heads per CTA (clusters of 4 x 16 warps)
int launch_dec_cluster_bf16_d512(const DecClusterP& p, cudaStream_t st);  // hidden 512, 8 heads x 64, filter 512 (SwinTRN decoder)
// stop-at-<EOS> instantiations of the four geometries (DecClusterP::lengths / work / eos): one launch for any batch
int launch_dec_cluster_bf16_eos(const DecClusterP& p, cudaStream_t st);
int launch_dec_cluster_bf16_d128_eos(const DecClusterP& p, cudaStream_t st);
int launch_dec_cluster_bf16_p2_eos(const DecClusterP& p, cudaStream_t st);
int launch_dec_cluster_bf16_d512_eos(const DecClusterP& p, cudaStream_t st);
void launch_cross_to_bf16(const float* src, __nv_bfloat16* kc, __nv_bfloat16* vc, int B, int S, int L, int Dm, int head_dim,
                          cudaStream_t st);

}  // namespace frx
