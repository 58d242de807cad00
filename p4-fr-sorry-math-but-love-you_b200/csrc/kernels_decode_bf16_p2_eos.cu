// Stop-at-<EOS> instantiation (FRX_DEC_EOS in kernels_decode_bf16.cu) of the two-heads-per-CTA geometry
// (kernels_decode_bf16_p2.cu).
#define FRX_DEC_D 256
#define FRX_DEC_FF 1024
#define FRX_DEC_HPC 2
#define FRX_DEC_KVDEPTH 2
#define FRX_DEC_NAME(x) x##_p2_eos
#define FRX_DEC_EOS 1
#define FRX_DEC_VARIANT 1
#include "kernels_decode_bf16.cu"
