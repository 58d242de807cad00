// Stop-at-<EOS> instantiation (FRX_DEC_EOS in kernels_decode_bf16.cu) of the EfficientSATRN geometry with one head
// per CTA: every row stops after the step that emits <EOS> and takes the next image of the batch.
#define FRX_DEC_D 256
#define FRX_DEC_FF 1024
#define FRX_DEC_NAME(x) x##_eos
#define FRX_DEC_EOS 1
#define FRX_DEC_VARIANT 1
#include "kernels_decode_bf16.cu"
