/*
 * melgan_b200.h -- C ABI of the B200-native MelGAN engine (libmelgan_b200.so).
 *
 * The reference (diver-j/melgan-multi) has no FFI or operator registry: its boundary for the
 * hot path is the torch.nn.Module protocol of models.py, imported by name at train.py:13
 * (`from models import Generator, MultiScaleDiscriminator, ...`).  This library sits directly
 * underneath a drop-in `models` module (melgan_multi_b200/models.py); each entry point below
 * names the reference code it replaces.  Plain pointers and sizes only, no torch types.
 *
 * Conventions
 *   - Every function returns 0 on success or a negative MG_ERR_* code; the message for the
 *     calling thread is available from mg_last_error_string().  Nothing throws or exits.
 *   - "device pointer" arguments are CUDA device addresses owned by the caller (PyTorch
 *     storage in practice); the library never frees or retains them past the call.
 *   - Tensors are fp32, contiguous, NCL ([batch][channel][length]) exactly like the
 *     reference's (models.py:61-71 takes [B,80,T], returns [B,1,256*T]).
 *   - `stream` is a cudaStream_t passed as void*; all work is enqueued asynchronously on it and
 *     the library never synchronises the device in the device-pointer entry points.
 *   - Re-entrant: no mutable global state except the thread-local error string.
 */
#ifndef MELGAN_B200_H_
#define MELGAN_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MG_OK 0
#define MG_ERR_INVALID_ARGUMENT (-1)
#define MG_ERR_CUDA (-2)
#define MG_ERR_UNSUPPORTED_DEVICE (-3)
#define MG_ERR_WORKSPACE_TOO_SMALL (-4)
#define MG_ERR_OUT_OF_MEMORY (-5)

#define MG_GEN_NUM_LAYERS 30 /* conv_pre, ups[0..3], 4 x (convs1[0..2], convs2[0..2]), conv_post */

/* ABI version of this header (bumped on any signature change). */
int mg_abi_version(void);

/* Message describing the last failure on the calling thread ("" if none). */
const char *mg_last_error_string(void);

/* 0 if the current CUDA device can run the sm_100a kernels, MG_ERR_UNSUPPORTED_DEVICE /
 * MG_ERR_CUDA otherwise.  There is no CPU fallback anywhere in this library. */
int mg_device_check(void);

/* ---------------------------------------------------------------------------------------
 * Weight-norm fold + packing.   Replaces: the weight_norm pre-forward hooks that recompute
 * w = g * v / ||v|| on every forward of every layer (models.py:16-28,46-59; 30 launches of
 * aten::_weight_norm_interface per Generator.forward, SURVEY 2.2) with ONE launch that folds
 * all 30 layers and writes them in the layouts the fused kernels stream from.
 *
 * v, g, bias: HOST arrays of MG_GEN_NUM_LAYERS DEVICE pointers in reference registration
 * order (conv_pre, ups.0-3, resblocks.0.convs1.0-2, resblocks.0.convs2.0-2, ..., conv_post);
 * shapes as in the reference state_dict (Conv1d weight_v [Cout,Cin,K], weight_g [Cout,1,1];
 * ConvTranspose1d weight_v [Cin,Cout,K], weight_g [Cin,1,1] -- the norm is per dim 0).
 * packed: device buffer of mg_gen_packed_bytes() bytes, 256-byte aligned.
 */
size_t mg_gen_packed_bytes(void);
int mg_gen_pack(const float *const *v, const float *const *g, const float *const *bias,
                void *packed, void *stream);

/* ---------------------------------------------------------------------------------------
 * Generator forward.   Replaces: models.Generator.forward (models.py:61-71): conv_pre, four
 * fused (LeakyReLU -> ConvTranspose1d -> ResBlock) stages (ResBlock.forward, models.py:32-40),
 * LeakyReLU -> conv_post -> tanh fused into the last stage.
 *
 * mel   [B, 80, T]     device, fp32
 * audio [B, 1, 256*T]  device, fp32
 * workspace: device scratch of at least mg_gen_workspace_bytes(B, T) bytes, 256-byte aligned.
 * Any B >= 1, T >= 1 (train.py:157 feeds whole utterances).
 */
size_t mg_gen_workspace_bytes(int B, int T);
int mg_gen_forward(const void *packed, const float *mel, float *audio, int B, int T,
                   void *workspace, size_t workspace_bytes, void *stream);

/* Ragged batch: mel [B, 80, T] padded, item b is its first lengths[b] frames (lengths: HOST array of B ints, each in
 * [1, T]).  audio [B, 1, 256*T]: audio[b, :, :256*lengths[b]] equals the forward of mel[b:b+1, :, :lengths[b]] alone, bit for
 * bit, and audio[b, :, 256*lengths[b]:] is exactly 0.  The padding frames of mel are never read (NaN there changes
 * nothing) and no result depends on earlier workspace contents.  workspace: mg_gen_workspace_bytes(B, T) bytes, as for
 * the uniform call; mg_gen_check_status(workspace, B, T, stream) reports on it.  Asynchronous on `stream` (no host
 * synchronisation, no allocation, no host-to-device copy: the per-item tables are kernel parameters), so the call can be
 * captured in a CUDA graph.  Only the frames that exist are computed: the batch slices are cut by cumulative frames.
 * Always runs the default kernel chain: mg_gen_set_pipeline / MG_GEN_TAIL (A/B knobs of the uniform call) do not apply.
 * Invalid arguments (lengths NULL, or a lengths[i] outside [1, T]) return MG_ERR_INVALID_ARGUMENT before any CUDA call;
 * the message names the index. */
int mg_gen_forward_varlen(const void *packed, const float *mel, float *audio, int B, int T, const int *lengths,
                          void *workspace, size_t workspace_bytes, void *stream);

/* Same as mg_gen_forward, but brackets each of the mg_gen_forward_launches() kernels with CUDA
 * events on `stream`, waits for the last one and returns the per-kernel device times in
 * kernel_ms[0 .. mg_gen_forward_launches()-1] (names: mg_gen_kernel_name(i)).  Used by bench.py for the
 * per-kernel roofline. */
int mg_gen_forward_timed(const void *packed, const float *mel, float *audio, int B, int T,
                         void *workspace, size_t workspace_bytes, void *stream, float *kernel_ms);

/* Waits for `stream` and reports whether the tensor-core pipeline of the last forward on `workspace`
 * completed (its producer/consumer waits are bounded so a logic error returns MG_ERR_CUDA here instead
 * of hanging the device). */
int mg_gen_check_status(const void *workspace, int B, int T, void *stream);

/* LeakyReLU -> ConvTranspose1d (models.py:64-65, ups[stage], models.py:48-51) on the tensor-core path:
 * x [B, 512>>stage, Lin] -> y [B, 256>>stage, S*Lin] (S = 8, 8, 2, 2), device fp32, x != y.  Synchronous;
 * parity-test entry point for the tcgen05 ConvT kernel. */
int mg_gen_convt(const void *packed, int stage, const float *x, float *y, int B, int Lin, void *stream);

/* One ResBlock (models.py:32-40) of stage `stage` (C = 256 >> stage channels) on the tensor-core path:
 * x, y [B, C, L] device fp32, x != y.  Synchronous; parity-test entry point for the tcgen05 kernel. */
int mg_gen_resblock(const void *packed, int stage, const float *x, float *y, int B, int L, void *stream);
/* Stage 2 or 3 as the pipeline runs it: LeakyReLU -> ConvTranspose1d(k4, s2) -> ResBlock in ONE kernel
 * (models.py:64-66); x [B][2C][Lin] is the previous stage's output, y [B][C][2 Lin] (C = 64 / 32).  Synchronous, like
 * mg_gen_resblock: a per-kernel parity entry point. */
int mg_gen_upres(const void *packed, int stage, const float *x, float *y, int B, int Lin, void *stream);

/* ResBlock `stage` (0..2) with the NEXT stage's LeakyReLU -> ConvTranspose1d fused at its tail, as the default pipeline runs it
 * (models.py:66 followed by :64-65 of the next loop iteration): x [B][C][L] is stage `stage`'s ConvT output, y
 * [B][C/2][S L] is stage+1's (S = 8 for stage 0, else 2).  Synchronous parity entry point. */
int mg_gen_resup(const void *packed, int stage, const float *x, float *y, int B, int L, void *stream);

/* conv_pre alone (models.py:46,62): mel [B,80,T] -> y [B,512,T], device fp32.  Synchronous parity-test entry point of
 * conv_rows_tc_kernel<80,512,k7>. */
int mg_gen_conv_pre(const void *packed, const float *mel, float *y, int B, int T, void *stream);
/* The last ResBlock with its fused epilogue (models.py:66-69 for stage 3: ResBlock -> LeakyReLU -> conv_post -> tanh):
 * x [B,32,L] (the stage-3 ConvT output) -> audio [B,1,L].  Synchronous parity-test entry point of the conv_post + tanh fusion. */
int mg_gen_resblock_post(const void *packed, const float *x, float *audio, int B, int L, void *stream);

/* Diagnostic twin of mg_gen_resblock: also returns 128 clock64 stamps (host buffer) of one interior CTA's
 * epilogue and MMA roles (slot meaning documented at the definition in csrc/mg_api.cu). */
int mg_gen_resblock_trace(const void *packed, int stage, const float *x, float *y, int B, int L, long long *trace_host);

/* Debug/parity tap: copies the activation after stage `which` (0 = conv_pre output [B,512,T],
 * 1..3 = ResBlock 0..2 output [B,C,L]; the last stage is fused with conv_post and has no tap) of the LAST mg_gen_forward that used `workspace` into
 * `out` (device, NCL).  Only valid immediately after that call on the same stream. */
int mg_gen_stage_output(const void *workspace, int which, float *out, int B, int T, void *stream);

/* ---------------------------------------------------------------------------------------
 * Multi-scale discriminator forward.   Replaces: models.MultiScaleDiscriminator.forward (models.py:119-135) and
 * Discriminator.forward (models.py:87-103) for a batch in which the caller has stacked real and generated audio
 * (Bt = 2B: every weight is streamed once for both; the reference calls d(y) and d(y_hat) separately), with the
 * AvgPool1d chain (models.py:114-117) fused into each scale's first conv and the 21 weight-norm folds done by one
 * mg_msd_pack launch.
 *
 * v, g, bias: HOST arrays of 21 DEVICE pointers, discriminator-major, layers in reference registration order
 *   (conv_pre, grouped_convs.0-3, conv_post1, conv_post2).
 * y [Bt, 1, L] device fp32.  fmaps: HOST array of 21 DEVICE pointers (scale-major, 7 per scale) receiving the feature
 *   maps [Bt, C_l, len] with len = lens[scale*7 + l] from mg_msd_lengths(L, lens); the first six of a scale are
 *   post-LeakyReLU, the seventh is conv_post2's raw output, i.e. the flattened logits [Bt, len].
 * status_word: >= 4 bytes of device memory; check it with mg_msd_check_status after the call (bounded waits).
 */
size_t mg_msd_packed_bytes(void);
int mg_msd_pack(const float *const *v, const float *const *g, const float *const *bias, void *packed, void *stream);
int mg_msd_lengths(int L, int *lens);
int mg_msd_forward(const void *packed, const float *y, int Bt, int L, float *const *fmaps, void *status_word, void *stream);
int mg_msd_check_status(const void *status_word, void *stream);

/* One stand-alone Discriminator (models.py:74-103: Discriminator() called on its own, outside MultiScaleDiscriminator):
 * v, g, bias: HOST arrays of 7 DEVICE pointers (conv_pre, grouped_convs.0-3, conv_post1, conv_post2); packed: device buffer of
 * mg_disc_packed_bytes() bytes, 256-byte aligned.  x [Bt,1,L] -> fmaps: HOST array of 7 DEVICE pointers, lengths
 * lens[0..6] of mg_msd_lengths(L, lens) (the scale-0 row); fmaps[6] is the flattened logits.  status_word as above. */
size_t mg_disc_packed_bytes(void);
int mg_disc_pack(const float *const *v, const float *const *g, const float *const *bias, void *packed, void *stream);
int mg_disc_forward(const void *packed, const float *x, int Bt, int L, float *const *fmaps, void *status_word, void *stream);

/* ---------------------------------------------------------------------------------------
 * Mel-spectrogram front end.   Replaces: mel_spectrogram (meldataset.py:44-55: zero-pad by (n_fft - hop)/2, librosa
 * melspectrogram with power 1 and Slaney-normalised triangles, log(clip(., 1e-5))) for the reference's analysis parameters
 * n_fft = 1024, hop = 256, win = 1024 (config.json:15-17), on the GPU: the loader's and the validation loop's librosa call
 * (train.py:164) without the host round trip.
 *   mg_mel_tables_build fills a HOST buffer of mg_mel_tables_bytes() bytes (window, twiddles, sparse filter bank);
 *     norm: 0 none, 1 Slaney area normalisation (= librosa 0.6/0.7 `norm=1`, today's `norm="slaney"`), 2 L1.  The caller
 *     copies it to device memory (16-byte aligned) once.
 *   mg_mel_spectrogram: audio [B][L] device fp32 in [-1, 1] -> mel [B][n_mels][T] device fp32, T = mg_mel_frames(L)
 *     (= L / 256 when L is a multiple of 256).  Asynchronous on `stream`.
 */
size_t mg_mel_tables_bytes(void);
int mg_mel_tables_build(int sampling_rate, int n_mels, float fmin, float fmax, int norm, void *tables_host);
int mg_mel_frames(int L);
int mg_mel_spectrogram(const void *tables, const float *audio, float *mel, int B, int L, void *stream);

/* ---------------------------------------------------------------------------------------
 * Host-buffer engine.   The call a non-PyTorch host makes: owns its device buffers, takes and
 * returns HOST memory, and performs the host<->device copies itself (this is the path
 * bench.py times as "e2e").  One engine per host thread / CUDA stream.
 */
typedef struct mg_gen_engine mg_gen_engine;

/* Creates an engine able to run up to max_B x max_T (it grows on demand if exceeded). */
int mg_gen_engine_create(mg_gen_engine **out, int max_B, int max_T);
/* v/g/bias: HOST arrays of 30 HOST pointers (state_dict tensors, reference order). */
int mg_gen_engine_load_state(mg_gen_engine *e, const float *const *v, const float *const *g,
                             const float *const *bias);
/* mel_host [B,80,T] -> audio_host [B,1,256T]; synchronous (returns when audio_host is filled).
 * Pinned host memory is used as given; pageable memory is staged through an internal pinned
 * buffer.  The copies are cut with the batch slices (mg_gen_forward_slices): a slice's audio goes
 * back to the host while the other slices are still computing. */
int mg_gen_engine_forward(mg_gen_engine *e, const float *mel_host, float *audio_host, int B, int T);
/* The ragged form (contract of mg_gen_forward_varlen; lengths: HOST array of B ints in [1, T]): mel_host [B,80,T] padded,
 * audio_host [B,1,256T] with exact zeros past each item's 256*lengths[b] samples.  Synchronous, like mg_gen_engine_forward. */
int mg_gen_engine_forward_varlen(mg_gen_engine *e, const float *mel_host, float *audio_host, int B, int T, const int *lengths);
/* Device time of the last forward in milliseconds (CUDA events on the engine's stream around the sliced
 * upload -> kernels -> download sequence). */
int mg_gen_engine_last_kernel_ms(mg_gen_engine *e, float *ms);
void mg_gen_engine_destroy(mg_gen_engine *e);

/* ---- discriminator backward (autograd of Discriminator.forward, models.py:87-103): no aten / cuDNN call is left --------
 * Conventions: dz = gradient w.r.t. a layer's PRE-activation output (i.e. already multiplied by LeakyReLU'), x = the layer's
 * input, dw = gradient of the layer's FOLDED weight in torch layout, db = bias gradient; mg_msd_wn_backward turns the layers'
 * dw into (d weight_v, d weight_g). */

/* The whole backward of discriminator `scale` in ONE call: the host side walks the seven layers from the logits down and
 * enqueues the kernels of the per-layer entry points below itself (what models._MSDFunction.backward uses).
 *   x0 [Bt][1][L0]: the discriminator's input (the pooled audio for scale > 0); fmap[7]: the maps the forward returned;
 *   gfmap[7]: gradient w.r.t. each returned map (NULL entries: none); gx0 [Bt][1][L0] or NULL (input gradient not needed);
 *   dw[7] / db[7]: outputs -- layers the gradient does not reach are left untouched and reported in reached[7] (host ints,
 *   may be NULL); workspace: bytes from the helper. */
size_t mg_msd_scale_backward_workspace_bytes(int Bt, int L0);
int mg_msd_scale_backward(const void *packed, int scale, const float *x0, const float *const *fmap, const float *const *gfmap,
                          float *gx0, float *const *dw, float *const *db, int *reached, void *workspace, size_t workspace_bytes,
                          int Bt, int L0, void *status_word, void *stream);

/* dz = (g1 + g2) * LeakyReLU'(out) over n elements (g2 may be NULL): the gradient entering a layer's pre-activation from the
 * next layer and from the feature-map loss, in one launch (F.leaky_relu backward of models.py:91,94,97 + the add). */
int mg_lrelu_backward(const float *g1, const float *g2, const float *out, float *dz, long long n, void *stream);

/* Gradients of ONE grouped conv (layer 1..4: k41, pad 20, 4 input channels per group, stride 4/4/4/1) of discriminator
 * `scale` of the packed MSD blob, each a single launch (cuDNN runs one kernel per group):
 *   dz [Bt][Cout][Lout], x [Bt][Cin][Lin]; dx [Bt][Cin][Lin] (NULL: skip), dw [Cout][4][41] + db [Cout] (dw NULL: skip both). */
size_t mg_msd_grouped_backward_workspace_bytes(int layer, int Bt, int Lout);
int mg_msd_grouped_backward(const void *packed, int scale, int layer, const float *dz, const float *x, float *dx, float *dw,
                            float *db, void *workspace, size_t workspace_bytes, int Bt, int Lin, int Lout, void *stream);

/* Data gradient of conv_post1 (Conv1d 1024 -> 1024, k5, pad 2; models.py:84,96) of discriminator `scale`: dz [Bt][1024][L]
 * -> dx [Bt][1024][L], on the same tcgen05 kernel as the forward, streaming the transposed, tap-flipped copy of the weights
 * that mg_msd_pack / mg_disc_pack keep for it. */
int mg_msd_post1_dgrad(const void *packed, int scale, const float *dz, float *dx, int Bt, int L, void *status_word, void *stream);
/* Weight and bias gradient of conv_post1 (no weights needed): x [Bt][1024][L], dz [Bt][1024][L] -> dw [1024][1024][5],
 * db [1024]; one tcgen05 launch, split-bf16 (fp32-grade) with fp32 accumulation over all Bt * L positions. */
int mg_msd_post1_wgrad(const float *x, const float *dz, float *dw, float *db, int Bt, int L, void *status_word, void *stream);

/* Backward of conv_pre (layer 0: Conv1d 1 -> 16, k15; x [Bt][1][L], dz [Bt][16][L], dw [16][1][15]) or conv_post2 (layer 6:
 * Conv1d 1024 -> 1, k3; x [Bt][1024][L], dz [Bt][1][L], dw [1][1024][3]) of discriminator `scale` (autograd of models.py:90,99):
 * dx (same shape as x; NULL: skip -- conv_pre's is only needed when the audio requires a gradient), dw, db.  fp32, fixed
 * summation order.  Layer 0 needs a workspace (bytes from the helper), layer 6 none. */
size_t mg_msd_edge_backward_workspace_bytes(int layer, int Bt, int L);
int mg_msd_edge_backward(const void *packed, int scale, int layer, const float *dz, const float *x, float *dx, float *dw, float *db,
                         void *workspace, size_t workspace_bytes, int Bt, int L, void *stream);

/* weight-norm backward of the 21 layers of an MSD blob in one launch: v, g, dw, dv, dg are HOST arrays of 21 device pointers
 * (dw[i] NULL: layer skipped):  dg = <dw, v> / |v|,  dv = (g / |v|) (dw - <dw, v> v / |v|^2) per norm row. */
int mg_msd_wn_backward(const float *const *v, const float *const *g, const float *const *dw, float *const *dv,
                       float *const *dg, void *stream);

/* ---- multi-tensor Adam (the optimizer step either side of the path: train.py:51-52,118,129) -------------------------
 * One launch updates `count` parameter tensors.  p, g, m, v: DEVICE arrays of `count` device pointers (parameter,
 * gradient, exp_avg, exp_avg_sq); n: DEVICE array of element counts; first: DEVICE array of count + 1 ints with
 * first[i] = sum_{j<i} ceil(n[j] / mg_adam_chunk()), total_ctas = first[count].  `step` is the 1-based step number of
 * this update.  Arithmetic of torch.optim.Adam (L2 weight decay, no amsgrad). */
int mg_adam_chunk(void);
int mg_adam_step(float *const *p, const float *const *g, float *const *m, float *const *v, const long long *n,
                 const int *first, int count, int total_ctas, float lr, float beta1, float beta2, float eps,
                 float weight_decay, long long step, void *stream);

/* ---- fused loss reductions (reference: feature_loss / discriminator_loss / generator_loss, models.py:138-167) ----
 * A loss is a table of `count` (<= 24) rows; out[i] = mean over the n[i] elements of
 *   mode 0: |a[i] - b[i]|   (one feature-map pair of feature_loss, models.py:142)
 *   mode 1: (1 - a[i])^2    (real term of discriminator_loss :151, generator_loss :165)
 *   mode 2: a[i]^2          (generated term of discriminator_loss :152)
 * (b[i] is ignored for modes 1, 2).  All rows are reduced by one launch plus a fixed-order combine (bit-reproducible);
 * `workspace` holds the per-CTA partial sums.  The caller scales / sums the row means (x10 for feature_loss).
 * mg_loss_backward writes grad_a[i] (and grad_b[i] for mode 0; either may be NULL) = grad_out[i] * d out[i] / d input;
 * grad_out is a DEVICE array of `count` floats. */
size_t mg_loss_workspace_bytes(const long long *n, int count);
int mg_loss_forward(const float *const *a, const float *const *b, const long long *n, const int *mode, int count,
                    float *out, void *workspace, size_t workspace_bytes, void *stream);
int mg_loss_backward(const float *const *a, const float *const *b, const long long *n, const int *mode, int count,
                     const float *grad_out, float *const *grad_a, float *const *grad_b, void *stream);

/* Number of kernels in the generator's chain (at most 16) and the name of the i-th one.  mg_gen_forward cuts
 * the batch into mg_gen_forward_slices(B, T) contiguous slices whose chains run concurrently on forked streams
 * (joined back into `stream` before it returns), so one forward enqueues slices x launches kernels. */
int mg_gen_forward_launches(void);
int mg_gen_forward_slices(int B, int T);
/* Selects the generator chain for the calling thread: bit i (1..3) of tail_mask = stage i's ConvT fused at the tail of
 * ResBlock i-1's kernel; 0 = one kernel per ConvT / ResBlock (all stage outputs materialised: mg_gen_stage_output works for
 * which = 1..3); -1 = the default (environment MG_GEN_TAIL, else all three).  For tests and A/B measurements. */
int mg_gen_set_pipeline(int tail_mask);
const char *mg_gen_kernel_name(int i);
/* Template configuration of the i-th chain kernel at T mel frames per item (e.g. "resblock_tc_kernel<RbCfg<128,2,4,4,1,0,0,1,0,1>>/NH4"):
 * profile evidence (profiles/ ncu captures) records it, and bench.py only quotes a capture taken with the configuration this
 * build actually runs. */
const char *mg_gen_kernel_config(int i, int T);

#ifdef __cplusplus
}
#endif
#endif /* MELGAN_B200_H_ */
