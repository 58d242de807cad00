// Stop-at-<EOS> instantiation (FRX_DEC_EOS in kernels_decode_bf16.cu) of the LiteSATRN geometry
// (kernels_decode_bf16_d128.cu).
#define FRX_DEC_D 128
#define FRX_DEC_FF 512
#define FRX_DEC_NAME(x) x##_d128_eos
#define FRX_DEC_EOS 1
#define FRX_DEC_VARIANT 1
#include "kernels_decode_bf16.cu"
