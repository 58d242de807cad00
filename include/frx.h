/*
 * frx.h -- C ABI of the B200-native formula-recognition hot path.
 *
 * The reference (bcaitech1/p4-fr-sorry-math-but-love-you) is pure Python/PyTorch
 * and has no FFI of its own, so these entry points are the ones its operator
 * API for this path would bind (SURVEY.md 8b).  Each one names the reference
 * interface it replaces (file:line under /root/reference).  Plain pointers and
 * sizes only -- no torch types cross this boundary.
 *
 * Conventions
 *   - every function returns 0 on success, non-zero on failure; the message is
 *     available from frx_last_error(h) (the Python host raises RuntimeError);
 *   - device pointers are caller-owned (torch storage), valid for the call,
 *     and all work is enqueued on the passed stream (a cudaStream_t passed as
 *     void*) -- no hidden synchronisation unless stated;
 *   - the handle owns packed weights, KV caches and workspaces;
 *   - one handle per (process, device); not thread-safe (the reference is
 *     single-threaded).
 */
#ifndef FRX_H_
#define FRX_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct frx_handle frx_handle;

enum { FRX_NET_EFFICIENT_SATRN = 0, FRX_NET_LITE_SATRN = 1, FRX_NET_SWIN = 2 };
enum { FRX_PREC_FP32 = 0, FRX_PREC_BF16 = 1 };
enum { FRX_DTYPE_F32 = 0, FRX_DTYPE_I64 = 1 };

/* Mirrors what the constructors read from FLAGS and the vocab:
 * networks/EfficientSATRN.py:664-692 (EfficientSATRN.__init__),
 * networks/LiteSATRN.py:548-576, networks/SWIN.py:1024-1049 (SWIN fixes the encoder to Swin-B/384:
 * height = width = 384, in_ch = 3, enc_hidden = 1024; the enc_* SATRN fields are ignored). */
typedef struct frx_config {
  int32_t network;      /* FRX_NET_* */
  int32_t height;       /* FLAGS.input_size.height */
  int32_t width;        /* FLAGS.input_size.width  */
  int32_t in_ch;        /* FLAGS.data.rgb */
  int32_t enc_hidden, enc_filter, enc_layers, enc_heads;          /* FLAGS.SATRN.encoder.* */
  int32_t dec_src, dec_hidden, dec_filter, dec_layers, dec_heads; /* FLAGS.SATRN.decoder.* */
  int32_t num_classes;  /* len(train_dataset.id_to_token) */
  int32_t sos_id, eos_id, pad_id;
  int32_t max_batch;    /* per-GPU image batch the workspaces are sized for */
  int32_t max_steps;    /* decode steps the KV cache is sized for (expected.size(1)-1) */
  int32_t precision;    /* FRX_PREC_* : arithmetic of the dense contractions / KV cache */
  int32_t device;       /* CUDA device ordinal */
} frx_config;

/* Library / build identification ("frx <ver> sm_100a"). */
const char* frx_version(void);

/* Replaces the nn.Module constructors (EfficientSATRN.py:664-695). */
int frx_create(const frx_config* cfg, frx_handle** out);
void frx_destroy(frx_handle* h);
const char* frx_last_error(const frx_handle* h);

/* Replaces nn.Module.load_state_dict (EfficientSATRN.py:694-695): call once per
 * state_dict entry with the reference's own key (SURVEY App. A.2).  `data` may
 * be a host or a device pointer (cudaMemcpyDefault); the library keeps its own
 * copy.  Also used for the three host-built positional tables that are NOT in
 * the state_dict (EfficientSATRN.py:95-99,404-405) under the reserved names
 * "pe2d.h" [h,C], "pe2d.w" [w,C], "pe1d" [500,D]. */
int frx_load_tensor(frx_handle* h, const char* name, const void* data,
                    const int64_t* shape, int32_t ndim, int32_t dtype);

/* Packs everything loaded so far into the kernels' layouts (eval-mode BN folded
 * to per-channel scale/shift, conv weights to [O][kh][kw][I], decoder linears
 * concatenated/transposed).  Fails if a tensor the network needs is missing or
 * has the wrong shape.  Must be called after the last frx_load_tensor and again
 * after any re-load. */
int frx_finalize_weights(frx_handle* h);

/* SATRNEncoder.forward (EfficientSATRN.py:311-323).
 * images  : device fp32 [B, in_ch, H, W] (NCHW, contiguous)
 * memory  : device fp32 [B, h*w, enc_hidden] (the reference's `src`, contiguous) */
int frx_encode(frx_handle* h, const float* images, int32_t batch, float* memory, void* stream);

/* SATRNDecoder.forward, inference branch (EfficientSATRN.py:528-566) followed by
 * decode()'s topk(1) (postprocessing/decoding.py:38-40).
 * memory  : device fp32 [B, h*w, dec_src]
 * logits  : device fp32 [B, steps, num_classes] or NULL
 * tokens  : device int64 [B, steps] or NULL
 * forced  : device int64 [B, steps] or NULL; when given, token t+1 fed to the
 *           decoder is forced[:, t] instead of the argmax (forced decoding,
 *           used by the parity tests; the reference's teacher_forcing_ratio=0
 *           loop is forced == NULL). */
int frx_decode_greedy(frx_handle* h, const float* memory, int32_t batch, int32_t steps,
                      float* logits, int64_t* tokens, const int64_t* forced, void* stream);

/* EfficientSATRN.forward(input, expected, is_train=False, ...) (EfficientSATRN.py:697-706):
 * encode + greedy decode with DEVICE buffers. */
int frx_forward_greedy(frx_handle* h, const float* images, int32_t batch, int32_t steps,
                       float* logits, int64_t* tokens, void* stream);

/* Greedy decode that stops each image at its first <EOS> (what id_to_string keeps, utils/utils.py:134-164), opt-in.
 * len[b] = index of the first emitted <EOS> + 1 (emitted: the arg-max, or with managed != 0 the DecodingManager's pick
 * -- the token frx_decode_greedy writes to `tokens`), or max_steps if there is none.  With `forced`, row b stops after
 * the step t at which forced[b, t] == <EOS> instead.
 * logits  : device fp32 [B, max_steps, num_classes] (managed: masked softmax rows) or NULL.  Rows t < len[b] are
 *           bit-identical to frx_decode_greedy's (frx_decode_greedy_managed's) on the same handle and batch; rows
 *           t >= len[b] are 0.
 * tokens  : device int64 [B, max_steps] or NULL: the full decode's tokens for t < len[b], <PAD> after.
 * lengths : device int32 [B].
 * Errors as frx_decode_greedy / frx_decode_greedy_managed (managed with forced is rejected).  The 16-bit persistent
 * decode kernel stops the work of an image at its <EOS> and hands its cluster row the next image; fp32 mode and 16-bit
 * handles on the step kernels decode all max_steps and apply the same contract afterwards (same output, no time saved).
 * Enqueues work only (no synchronisation), so it can be captured in a CUDA graph. */
int frx_decode_greedy_eos(frx_handle* h, const float* memory, int32_t batch, int32_t max_steps, float* logits,
                          int64_t* tokens, int32_t* lengths, const int64_t* forced, int32_t managed, void* stream);
/* frx_encode + frx_decode_greedy_eos. */
int frx_forward_greedy_eos(frx_handle* h, const float* images, int32_t batch, int32_t max_steps, float* logits,
                           int64_t* tokens, int32_t* lengths, int32_t managed, void* stream);

/* Same call with HOST buffers (pinned or pageable): H2D of the images, encode,
 * decode, D2H of tokens (and of logits when logits_host != NULL); synchronises
 * the stream before returning.  This is the end-to-end entry bench.py times. */
int frx_forward_greedy_host(frx_handle* h, const float* images_host, int32_t batch, int32_t steps,
                            float* logits_host, int64_t* tokens_host, void* stream);

/* The same entry, pipelined over consecutive batches (an inference loop over a DataLoader, inference_single.py:50-61):
 * _submit enqueues H2D (own stream) -> encode + decode (`stream`) -> D2H of the tokens (own stream) for one of two slots
 * and returns at once; _wait blocks until that slot's tokens are in tokens_host.  With two batches in flight the copies
 * of batch i +- 1 run under the compute of batch i.  The host buffers must stay valid (and should be pinned) until _wait. */
int frx_forward_greedy_host_submit(frx_handle* h, const float* images_host, int32_t batch, int32_t steps,
                                   int64_t* tokens_host, int32_t slot, void* stream);
int frx_forward_greedy_host_wait(frx_handle* h, int32_t slot);

/* EfficientSATRN_decoder.reset_status / step_forward (EfficientSATRN.py:932-952),
 * the stateful API the ensemble driver uses (utils/ensemble_utils.py:83-118).
 * frx_decode_begin projects the cross-attention K/V of `memory` once and
 * resets step_idx; frx_decode_step consumes target [B] int64 and writes
 * logits [B, num_classes] for position step_idx, then increments it. */
int frx_decode_begin(frx_handle* h, const float* memory, int32_t batch, void* stream);
int frx_decode_step(frx_handle* h, const int64_t* target, float* logits, void* stream);

/* Image input pipeline on the device (data/dataset.py:62-83, data/augmentations.py:27-46): for `batch` decoded uint8
 * images (HWC, tightly packed one after another in the device buffer `packed`; offsets / heights / widths are HOST
 * arrays) -> optional 90-degree rotation of tall images (h / w > 2), cv2.resize(INTER_LINEAR) to out_h x out_w (OpenCV's
 * 8-bit fixed-point arithmetic, bit for bit), (x - mean * 255) * (1 / (std * 255)), HWC -> CHW: out fp32
 * [batch, channels, out_h, out_w] on the device -- the tensor EfficientSATRN.forward takes.  No handle: stateless.
 * Returns 0, 1 (bad argument), 2 (allocation / copy failed), 3 (launch failed). */
int frx_preprocess_u8(const uint8_t* packed, const int64_t* offsets, const int32_t* heights, const int32_t* widths,
                      int32_t batch, int32_t channels, int32_t out_h, int32_t out_w, const float* mean, const float* stddev,
                      int32_t rotate_tall, float* out, void* stream);

/* Ensemble decoding, utils/ensemble_utils.py:71-118 (make_decoder_values): n_models decoder handles advance in lock
 * step; per step every model's step_forward logits are soft-maxed and averaged (:95-105), the average optionally goes
 * through DecodingManager.sift (:107-108; rule tables of handles[0], frx_set_decoding_rules), its arg-max is the next
 * target of every model (:110).  memories[m]: model m's encoder output [B, S, C] (device).  probs [B, steps, V]: the
 * stacked distributions (:112-115); tokens [B, steps] (optional): their arg-max.  All handles on one device. */
int frx_ensemble_decode(frx_handle* const* handles, int32_t n_models, const float* const* memories, int32_t batch,
                        int32_t steps, float* probs, int64_t* tokens, int32_t use_manager, void* stream);

/* EfficientSATRN.beam_search (EfficientSATRN.py:708-867) with topk=1 via
 * decode(method="beam") (postprocessing/decoding.py:42-48): per-sample
 * best-first search, score -logp/len in fp64 (decoding.py:80), node order on
 * len (decoding.py:83-87), budget (max_sequence-1) expansions, stop at the
 * first popped EOS, rows start with SOS and are PAD-padded.
 * tokens  : device int64 [B, max_sequence] */
int frx_beam_search(frx_handle* h, const float* memory, int32_t batch, int32_t beam_width,
                    int32_t max_sequence, int64_t* tokens, void* stream);

/* SATRNDecoder.forward, teacher-forced branch (EfficientSATRN.py:488-495) in
 * eval mode (dropout = identity).  In bf16 mode every linear layer (M = B*L rows) and the vocabulary
 * projection run on the tcgen05 GEMM (bf16 operands, fp32 accumulation / residual stream / LayerNorm).
 * text    : device int64 [B, L] (= expected[:, :-1])
 * logits  : device fp32 [B, L, num_classes] */
int frx_decode_teacher_forced(frx_handle* h, const float* memory, const int64_t* text,
                              int32_t batch, int32_t length, float* logits, void* stream);

/* DecodingManager (postprocessing/postprocessing.py:182-405; built by get_decoding_manager, :158-180, and attached
 * to the model by inference_single.py:80-95): rule-constrained greedy decoding.  The host compiles the manager's
 * `rules` dict against its `tokens` list into per-class tables:
 *   flags[v] : bit 0 cannot_initial, 1 next_underbar, 2 next_lbracket, 3 cannot_next_underbar, 4 cannot_next_lbracket
 *   limit[v] : limit_params[token] where limit_series[token] is true, else 0
 *   ids6     : ids of "<SOS>", "<EOS>", "" (the empty token), "{", "}", "_"
 * Host pointers; the library keeps device copies. */
int frx_set_decoding_rules(frx_handle* h, const int32_t* flags, const int32_t* limit, int32_t num_classes,
                           const int32_t* ids6);

/* SATRNDecoder.forward inference branch with a manager attached (EfficientSATRN.py:536-564): every step's logits
 * row goes through DecodingManager.sift (:193-233) -- softmax, black-listed classes (MemoryNode._look_back,
 * :327-391) zeroed, argmax = next input token, MemoryNode.record (:303-325).
 * probs   : device fp32 [B, steps, num_classes] MASKED SOFTMAX rows (what the reference's forward returns) or NULL
 * tokens  : device int64 [B, steps] or NULL
 * (The reference itself raises TypeError after its last step: it calls manager.reset() without the required
 * argument, :564 vs postprocessing.py:237.  These entry points return the loop's results.)
 * The step kernels are the fp32 ones in either precision mode. */
int frx_decode_greedy_managed(frx_handle* h, const float* memory, int32_t batch, int32_t steps, float* probs,
                              int64_t* tokens, void* stream);
int frx_forward_greedy_managed(frx_handle* h, const float* images, int32_t batch, int32_t steps, float* probs,
                               int64_t* tokens, void* stream);

/* Introspection for bench.py / tests: number of kernel launches the library
 * has enqueued since creation (nodes of replayed CUDA graphs included), and the
 * bytes currently allocated by the handle. */
int64_t frx_launch_count(const frx_handle* h);
int64_t frx_device_bytes(const frx_handle* h);

/* Debug taps used by the parity tests: copy an internal activation (NHWC fp32)
 * produced by the last frx_encode into `out` (device).  Names: "stem",
 * "eff_block.<s>.<i>", "trunk", "pe2d", "enc_layer<i>".  Returns the number of
 * floats written through *count.  Only available when the handle was created
 * with taps enabled via frx_set_option(h, "taps", 1).
 *
 * frx_set_option keys (test / bench switches; defaults in parentheses):
 *   "taps" (0)      keep per-block activations for frx_read_tap
 *   "graphs" (1)    fp32 mode: replay the greedy loop as a CUDA graph
 *   "timing" (0)    record CUDA events for frx_last_timing
 *   "prof" (0)      in-kernel stage profiler of the bf16 decode kernel (frx_read_prof)
 *   "parts" (3)     bit 0 encoder, bit 1 decoder (EfficientSATRN_encoder / _decoder handles); re-finalize after changing
 *   "enc_fp32" (0)  bf16 mode: run the encoder on the fp32 kernels
 *   "train_splitk" (1)  training step: GEMM launches of few output tiles (squeeze-excite FCs, late-stage 1x1 convolutions
 *                       of a 16-image batch) split K over CTAs; partials are summed in split order by a second kernel (no
 *                       atomics).  0 = one pass over K per tile
 *   "tc_ws" (1), "tc_im2col" (1), "conv24" (1)   bf16 encoder: persistent warp-specialised tcgen05 GEMM / TMA-im2col feed /
 *                   halo-tile kernel for the 24-channel convs; 0 selects the variant each one replaced
 *   "dec_hpc" (0)   bf16 decode, 256-wide decoder: heads per CTA (1: clusters of 8, 2: clusters of 4); 0 = by batch size */
int frx_set_option(frx_handle* h, const char* key, int64_t value);
int frx_read_tap(frx_handle* h, const char* name, float* out, int64_t capacity, int64_t* count,
                 int32_t* shape4, void* stream);

/* Times (milliseconds, CUDA events on the launching stream) of the phases of the
 * last frx_forward_greedy* call when option "timing" is 1: [0]=encode,
 * [1]=cross-KV + decode loop, [2]=total, [3]=the persistent decode kernel alone
 * (bf16 mode; 0 otherwise). */
int frx_last_timing(const frx_handle* h, float* ms4);

/* Test / micro-benchmark hook: the tcgen05 implicit-GEMM kernel on its own.
 * C[M,N] = act((A * W^T) * scale + shift); A bf16 [M,K] (dense) or, when conv7 !=
 * NULL, an NHWC bf16 activation gathered as a k x k convolution with conv7 =
 * {B, H, W, Cin, k, stride, tf_same_padding}; W bf16 [N,K]; C bf16 or fp32. */
int frx_tc_gemm(frx_handle* h, const void* A, const void* W, void* C, int32_t M, int32_t N, int32_t K,
                const int32_t* conv7, const float* scale, const float* shift, int32_t act, int32_t out_f32,
                void* stream);

/* Per-stage SM-cycle totals of the last bf16 decode kernel (option "prof" = 1;
 * recorded by one thread of cluster 0): 16 counters, see DESIGN.md. */
int frx_read_prof(frx_handle* h, int64_t* out16);

/* ---------------------------------------------------------------------------------------------------------------
 * Training step (EfficientSATRN, and LiteSATRN -- the student of train_modules/train_distillation.py:95-117, networks/
 * LiteSATRN.py:21-70, :581-590): one iteration of train_modules/train_single_opt.py:72-112 --
 *   model.train(); output = model(input, expected, True, 1.0)   (teacher forcing, EfficientSATRN.py:488-495, :697-706;
 *                                                                BatchNorm batch statistics)
 *   loss = CrossEntropyLoss(ignore_index=PAD)(output.transpose(1, 2), expected[:, 1:])   (:82-86, EfficientSATRN.py:690-692)
 *   loss.backward(); clip_grad_norm_(params, max_grad_norm); AdamW.step()                (:92-98, utils/utils.py:91-92)
 * fp32 like the reference (no autocast).  Dropout is off unless frx_train_set_dropout enables it.
 *
 * frx_train_create      copies the loaded parameters into the training state (one flat fp32 buffer in kernel layouts, a
 *                       parallel gradient buffer, Adam moments, BatchNorm running statistics) and sizes the activation
 *                       tape for max_batch images and targets of max_len tokens.  grad_buffer: caller-owned device
 *                       buffer of frx_train_param_count floats to hold the gradients (e.g. a torch tensor the host
 *                       all-reduces with NCCL), or NULL to let the library allocate it.
 * frx_train_fwd_bwd     images fp32 [B, in_ch, H, W], expected int64 [B, len_plus_1] (PAD-padded, as the reference's
 *                       d["truth"]["encoded"] with -1 replaced by PAD, :77-78) -> gradients in the flat buffer,
 *                       *loss_out (host or device float) = the mean loss over the non-PAD targets.  While the backward
 *                       pass runs, the bucket callback (if set) is invoked on the calling thread as soon as every kernel
 *                       contributing to a contiguous range [offset, offset + count) of the gradient buffer has been
 *                       enqueued on `stream`, so the host can start that range's all-reduce under the rest of the pass.
 * frx_train_apply       gradient *= grad_scale (1 / world size after a sum all-reduce); norm = ||g||_2;
 *                       g *= min(1, max_grad_norm / (norm + 1e-6)); AdamW(lr, betas (0.9, 0.999), eps 1e-8,
 *                       weight_decay).  *grad_norm_out (host or device float) = norm before clipping.
 * frx_train_export      parameter or BatchNorm running statistic by its state_dict name -> dst in the reference's
 *                       state_dict layout (host or device pointer).  frx_train_read_grad: the same for gradients. */
int frx_train_create(frx_handle* h, int32_t max_batch, int32_t max_len, float* grad_buffer);
void frx_train_destroy(frx_handle* h);
int64_t frx_train_param_count(frx_handle* h);
int frx_train_fwd_bwd(frx_handle* h, const float* images, const int64_t* expected, int32_t batch, int32_t len_plus_1,
                      float* loss_out, void* stream);
/* The same pass in two calls, for callers that compute the loss themselves (the reference's loop: output = model(...);
 * loss = criterion(output.transpose(1, 2), expected[:, 1:]); loss.backward() -- train_single_opt.py:79-92):
 * frx_train_forward  train-mode forward (BatchNorm batch statistics, running statistics updated) -> logits [B, L, V]
 *                    (loss_out optional: the CrossEntropy(ignore PAD) of the same pass);
 * frx_train_backward continues from the logits gradient [B, L, V] the caller's criterion produced and leaves the
 *                    parameter gradients in the flat buffer / frx_train_read_grad.  images: the forward call's.
 * frx_train_import   overwrite one parameter of the training state from the state_dict layout (an external optimiser
 *                    stepped the nn.Parameters). */
int frx_train_forward(frx_handle* h, const float* images, const int64_t* expected, int32_t batch, int32_t len_plus_1,
                      float* logits_out, float* loss_out, void* stream);
int frx_train_backward(frx_handle* h, const float* images, const float* dlogits, int32_t batch, int32_t len_plus_1, void* stream);
int frx_train_import(frx_handle* h, const char* name, const float* src);
int frx_train_grad_buffer(frx_handle* h, float** grads, int64_t* count);
int frx_train_set_bucket_callback(frx_handle* h, void (*callback)(void* ctx, int64_t offset, int64_t count), void* ctx);
int frx_train_apply(frx_handle* h, float lr, float weight_decay, float max_grad_norm, float grad_scale,
                    float* grad_norm_out, void* stream);
/* The dual-optimizer loop (train_modules/train_dual_opt.py:95-112): clip_grad_norm_ and AdamW separately over
 * model.encoder.parameters() (enc_lr) and model.decoder.parameters() (dec_lr). */
int frx_train_apply_dual(frx_handle* h, float enc_lr, float dec_lr, float weight_decay, float max_grad_norm, float grad_scale,
                         float* enc_grad_norm_out, float* dec_grad_norm_out, void* stream);
int frx_train_export(frx_handle* h, const char* name, float* dst);
int frx_train_read_grad(frx_handle* h, const char* name, float* dst);
int64_t frx_train_step_count(const frx_handle* h);
/* Debug view into the tape of the last frx_train_fwd_bwd call (what a forward/backward hook on the reference module
 * would see): copies the named buffer to dst (host or device, capacity floats) and returns its length; dst = NULL only
 * returns the length; -1 = unknown name.  Names: "dec<l>.d_linear0", "dec<l>.d_linear1", "dec<l>.d_ffn_out", ... */
int64_t frx_train_read_tap(frx_handle* h, const char* name, float* dst, int64_t capacity);
/* Dropout in the training pass (off after frx_train_create; p = p_ffn = 0 turns it off again).  p is the rate of the
 * reference's sites (FLAGS.dropout_rate): the 2-D PE output, the attention probabilities and the MHA outputs of every
 * encoder and decoder layer, the decoder input; p_ffn the rate after each ReLU of the decoder feed-forward blocks (0.1 in
 * the reference whatever the flag says).  Masks come from Philox4x32-10 with key = seed (low word, high word) and counter
 * (element index / 4, site + 16 * layer, step, rank), element index in the reference's layout of the site; step counts
 * the forward passes since frx_train_create, rank is the data-parallel rank.  An element is kept iff its word is
 * >= min(2^32 - 1, floor(p * 2^32)) (p as this float, computed in double); kept values are multiplied by
 * 1.0f / (1.0f - p).  The backward pass regenerates the masks of the forward pass it continues.  Rates outside [0, 1)
 * and a handle without training state are rejected.  Inference never applies dropout. */
int frx_train_set_dropout(frx_handle* h, float p, float p_ffn, uint64_t seed, int32_t rank);
/* Test hook: Philox4x32-10 of one counter and key, computed on the GPU by the function the dropout kernels use
 * (synchronous, host in and out). */
int frx_philox4x32(const uint32_t ctr[4], const uint32_t key[2], uint32_t out[4]);

#ifdef __cplusplus
}
#endif
#endif /* FRX_H_ */
