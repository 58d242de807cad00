// Stop-at-<EOS> instantiation (FRX_DEC_EOS in kernels_decode_bf16.cu) of the SwinTRN decoder geometry
// (kernels_decode_bf16_d512.cu).
#define FRX_DEC_D 512
#define FRX_DEC_FF 512
#define FRX_DEC_HD 64
#define FRX_DEC_MINBLOCKS 1
#define FRX_DEC_NAME(x) x##_d512_eos
#define FRX_DEC_EOS 1
#define FRX_DEC_VARIANT 1
#include "kernels_decode_bf16.cu"
