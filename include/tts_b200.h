/* tts_b200 -- C ABI of the B200-native (sm_100a) VITS + HiFiGAN inference hot path.
 *
 * The reference (coqui-ai/TTS v0.22.0) has no FFI for this path: its "operator API" is Python
 * classes + state_dict (SURVEY.md section 8b).  Each entry point below replaces the body of one
 * reference call; the Python mirror in tts_b200/ binds them with ctypes and keeps the reference's
 * class / function signatures.  INTEGRATION.md shows the binding a maintainer would add.
 *
 * Conventions
 *   - every function returns 0 on success, non-zero on error (1 = bad argument, 2 = CUDA error);
 *     b200tts_last_error() returns a thread-local message.  Nothing throws across the ABI.
 *   - tensors are raw DEVICE pointers, fp32 unless stated, in the reference's layouts
 *     ([B, C, T] with T contiguous); the caller owns every buffer.
 *   - *_create() takes HOST pointers to fp32 weights in PyTorch layout (weight-norm already
 *     folded: w = g * v / ||v||), packs them for the kernels and uploads them once.
 *   - scratch comes from a caller workspace sized by *_workspace_bytes(); handles are immutable
 *     after creation and may be shared by concurrent streams (each with its own workspace).
 *   - `stream` is a cudaStream_t passed as void*.
 */
#ifndef TTS_B200_H
#define TTS_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* Numerical precision of the tensor-core conv layers (the `precision` argument of the *_create_ex calls).
 *   B200TTS_PRECISION_FP32 (the default of every other create call): 3xTF32.  Both operands are split into
 *     hi + lo TF32 parts and each tap issues lo*hi + hi*lo + hi*hi, accumulated in fp32: within ~1e-5 relative RMS of
 *     an fp32 computation per layer, and the HiFiGAN waveform within 1e-4 RMS of the fp32 reference.
 *   B200TTS_PRECISION_TF32: single-pass TF32, the numerics PyTorch's cuDNN convolutions use by default
 *     (torch.backends.cudnn.allow_tf32).  Activations (after the leaky ReLU) and weights are rounded to TF32 -- to
 *     nearest, ties away from zero -- and each tap is one MMA accumulated in fp32.  Per output element the error is
 *     at most about (2^-10 + Cin*K*2^-23) * sum|w||x| plus the fp32 epilogue's roundings; measured on a B200:
 *     1e-4 to 3e-4 relative RMS per layer, 2e-4 to 5e-4 on the HiFiGAN waveform (cuDNN's TF32 on the same inputs:
 *     about 8e-4).  Faster: a third of the MMAs and of the operand bytes in shared memory, half the weight bytes.
 * Layers that do not run on the tensor cores (HiFiGAN conv_post and cond_layer, anything narrower than 32 rows, and
 * every layer created with allow_tensor_cores = 0) are exact FP32 in both modes.  Results are deterministic in both:
 * identical calls give identical bits, and a ragged call equals the dense one on every valid sample. */
#define B200TTS_PRECISION_FP32 0
#define B200TTS_PRECISION_TF32 1

const char* b200tts_last_error(void);
/* number of kernels launched by this library in this process (bench.py "gpu_launches") */
unsigned long long b200tts_launch_count(void);
int b200tts_version(void);
/* 1 if a tcgen05 conv launch (on any device of this process) ever hit a pipeline timeout.  The flag lives in mapped
 * host memory: no synchronisation here (call after a stream sync to cover the launches before it).  Every later
 * conv launch on that device also checks it and returns status 1, so a timeout cannot pass silently. */
int b200tts_debug_tc_error(void);

/* Debug / test aids: record, on the calling thread, which kernel family every conv launch dispatched to.
 * ids: 0 FP32-FMA tile kernel, 1 tcgen05 v1, 2 tcgen05 v2 (M = time), 3 tcgen05 v3 (M = rows), 4 v3 + staged epilogue,
 *      5 v3 grouped (narrow layers), 6 single-row streaming kernel (conv_post), 7 fused ResBlock kernel,
 *      8 v3 single-pass TF32, 9 v3 grouped single-pass TF32. */
void b200tts_debug_dispatch_begin(void);
int b200tts_debug_dispatch_end(int32_t* ids, int cap); /* returns the number of launches recorded */

/* ---- one conv layer with the fused prologue / epilogue the engines use -------------------------
 * The building block every dense contraction of the path runs on; replaces one
 * F.conv1d / F.conv_transpose1d call together with the element-wise ops around it, e.g. the ResBlock1 step
 * `xt = F.leaky_relu(x, 0.1); xt = c1(xt)` ... `x = xt + x` (TTS/vocoder/models/hifigan_generator.py:93-99) or
 * `o = self.ups[i](F.leaky_relu(o, 0.1))` (:248-249):
 *   y = ((conv(leaky_relu(x, in_slope)) + bias) + residual) * scale [+ y_old if accumulate] / post_div
 * weight: host, PyTorch layout ([Cout,Cin,K], or [Cin,Cout,K] when transposed); bias host or NULL; x [B,Cin,T],
 * residual / y [B,Cout,Tout] device.  in_slope = 1 disables the prologue.  allow_tensor_cores != 0 opts the layer into
 * the tcgen05 3xTF32 kernels (the decoder / flow setting); 0 keeps it on the exact FP32-FMA kernel (text encoder).
 */
typedef struct {
    int in_channels, out_channels, kernel_size, dilation, padding;
    int transposed; /* 1: ConvTranspose1d with `stride` (dilation must be 1) */
    int stride;
} b200tts_conv1d_config;
typedef struct b200tts_conv1d b200tts_conv1d;
int b200tts_conv1d_create(const b200tts_conv1d_config* cfg, const float* weight, const float* bias,
                          int allow_tensor_cores, b200tts_conv1d** out);
/* the same with an explicit B200TTS_PRECISION_* for the tensor-core kernels (b200tts_conv1d_create = FP32);
 * an unknown precision returns 1 */
int b200tts_conv1d_create_ex(const b200tts_conv1d_config* cfg, const float* weight, const float* bias,
                             int allow_tensor_cores, int precision, b200tts_conv1d** out);
void b200tts_conv1d_destroy(b200tts_conv1d* h);
int b200tts_conv1d_out_len(const b200tts_conv1d* h, int T);
int b200tts_conv1d_forward(const b200tts_conv1d* h, const float* x, int B, int T, float in_slope, const float* residual,
                           float scale, int accumulate, float post_div, float* y, void* stream);

/* ---- monotonic alignment search ------------------------------------------------------------
 * Replaces maximum_path_c / maximum_path_each, TTS/tts/utils/monotonic_align/core.pyx:11-47
 * (called through TTS/tts/utils/helpers.py:172-194 from Vits.forward_mas, vits.py:919).
 * value [B,Tx,Ty] f32 (NOT modified, unlike the reference's in-place DP); mask [B,Tx,Ty] f32 or
 * NULL (when given, value*mask is formed on load exactly like helpers.py:184); t_x,t_y int32 [B]
 * device pointers; path [B,Tx,Ty] written in full (zeros and ones) as int32 (path_is_f32 = 0,
 * the reference dtype, core.pyx:11) or float32 (path_is_f32 = 1, the dtype helpers.py:194 casts to).
 */
size_t b200tts_mas_workspace_bytes(int B, int Tx, int Ty);
int b200tts_mas(const float* value, const float* mask, const int32_t* t_x, const int32_t* t_y, int B, int Tx,
                int Ty, void* path, int path_is_f32, void* workspace, size_t workspace_bytes, void* stream);

/* Alignment straight from the prior statistics: replaces the body of Vits.forward_mas up to `attn`
 * (TTS/tts/models/vits.py:909-919): logp[b,x,y] = sum_c exp(-2 logs_p)(-0.5 z_p^2) + sum_c (m_p exp(-2 logs_p)) z_p
 * + sum_c(-0.5 log 2pi - logs_p) + sum_c(-0.5 m_p^2 exp(-2 logs_p)), then maximum_path(logp, mask) with
 * t_x / t_y = the lengths the masks encode.  z_p [B,C,Ty], m_p / logs_p [B,C,Tx]; path as b200tts_mas; logp_out
 * (nullable) [B,Tx,Ty] receives the log-likelihoods (otherwise they live in the workspace only). */
size_t b200tts_mas_from_stats_workspace_bytes(int B, int Tx, int Ty);
int b200tts_mas_from_stats(const float* z_p, const float* m_p, const float* logs_p, const int32_t* t_x, const int32_t* t_y,
                           int B, int C, int Tx, int Ty, void* path, int path_is_f32, float* logp_out, void* workspace,
                           size_t workspace_bytes, void* stream);

/* ---- HiFiGAN generator -----------------------------------------------------------------------
 * Replaces HifiganGenerator.forward, TTS/vocoder/models/hifigan_generator.py:236-265
 * (ctor arguments :163-178).
 * weights (host pointers, PyTorch layouts), in this order:
 *   conv_pre.w [C0,Cin,7], conv_pre.b [C0]
 *   cond_layer.w [C0,cond,1], cond_layer.b [C0]                      (only if cond_channels > 0)
 *   for each upsample stage s:
 *     ups[s].w [Cs_in, Cs_in/2, k] (ConvTranspose1d layout), ups[s].b
 *     for each resblock kernel j, for each dilation n:
 *       type "1": convs1[n].w, convs1[n].b, convs2[n].w, convs2[n].b
 *       type "2": convs[n].w,  convs[n].b
 *   conv_post.w [Cout, Clast, 7], conv_post.b (NULL pointer when conv_post_bias=False)
 */
typedef struct {
    int in_channels;
    int out_channels;
    int upsample_initial_channel;
    int cond_channels;
    int resblock_type; /* 1 or 2 */
    int num_upsamples;
    int upsample_factors[8];
    int upsample_kernel_sizes[8];
    int num_kernels;
    int resblock_kernel_sizes[8];
    int num_dilations;
    int resblock_dilations[8][8];
} b200tts_hifigan_config;

typedef struct b200tts_hifigan b200tts_hifigan;
int b200tts_hifigan_create(const b200tts_hifigan_config* cfg, const float* const* weights, int num_weights,
                           b200tts_hifigan** out);
/* the same with an explicit B200TTS_PRECISION_* for conv_pre, the upsamplers and the ResBlock convs
 * (b200tts_hifigan_create = FP32); an unknown precision returns 1.  b200tts_hifigan_precision: the handle's mode
 * (-1 for NULL). */
int b200tts_hifigan_create_ex(const b200tts_hifigan_config* cfg, const float* const* weights, int num_weights,
                              int precision, b200tts_hifigan** out);
int b200tts_hifigan_precision(const b200tts_hifigan* h);
void b200tts_hifigan_destroy(b200tts_hifigan* h);
size_t b200tts_hifigan_workspace_bytes(const b200tts_hifigan* h, int B, int T);
int b200tts_hifigan_out_len(const b200tts_hifigan* h, int T);
/* x [B,Cin,T]; g [B,cond,1] or NULL; wav [B,Cout,out_len(T)] */
int b200tts_hifigan_forward(const b200tts_hifigan* h, const float* x, const float* g, int B, int T, float* wav,
                            void* workspace, size_t workspace_bytes, void* stream);

/* b200tts_hifigan_forward with two optional extras (either may be NULL):
 *  - frame_lengths, device int32 [B]: valid frames per row of a padded batch.  Padded frames are then neither computed nor
 *    read: every launch stops a layer-specific margin past a row's end (the receptive field of the layers that still
 *    follow; b200tts_hifigan_margin_frames() is the largest, at the input rate), so every sample below
 *    frame_lengths[b] * prod(upsample_factors) is BIT-IDENTICAL to the dense call and the rest of the row is zero
 *    (the dense call, like the reference, fills it with the network's response to zero input, which no caller keeps).
 *  - peak_bits: conv_post's store folds max|wav| over everything it writes into *peak_bits (atomicMax on the float's
 *    bit pattern; the caller zeroes the word first, several calls may share it): the first half of save_wav's peak
 *    normalisation, TTS/utils/audio/numpy_transforms.py:439, without another pass. */
int b200tts_hifigan_forward_ex(const b200tts_hifigan* h, const float* x, const float* g, int B, int T, float* wav,
                               const int32_t* frame_lengths, uint32_t* peak_bits, void* workspace, size_t workspace_bytes,
                               void* stream);
int b200tts_hifigan_margin_frames(const b200tts_hifigan* h);

/* ---- hand-off around a standalone vocoder ---------------------------------------------------------
 * b200tts_vocoder_input replaces, in one pass on the device, what Synthesizer.tts does on the host between the TTS
 * model and the vocoder (TTS/utils/synthesizer.py:412-429):
 *   tts_ap.denormalize (TTS/utils/audio/processor.py:303-337)  ->  vocoder_ap.normalize (:259-301)
 *   -> interpolate_vocoder_input (TTS/vocoder/utils/generic_utils.py:11-29; bilinear, align_corners=False,
 *      recompute_scale_factor=True, scale [1, scale_factor])   -> replicate padding of HifiganGenerator.inference
 *      (TTS/vocoder/models/hifigan_generator.py:281)
 * x is addressed as x[b*x_batch_stride + c*x_channel_stride + t*x_time_stride] (the TTS model's [B,T,C] output or a
 * [B,C,T] spectrogram alike); y is [B, C, y_pitch] with b200tts_vocoder_input_len(T, scale_factor, padding) valid
 * columns per row (give y_pitch a multiple of 4 for the tensor-core kernels).  scaler_mean / scaler_scale: DEVICE
 * pointers to the [C] statistics of a mean-var AudioProcessor (stats_path), NULL otherwise.
 * b200tts_absmax / b200tts_to_int16: save_wav's `wav * (32767 / max(0.01, max|wav|))` -> int16
 * (TTS/utils/audio/numpy_transforms.py:439-441); *peak_bits as above.
 */
typedef struct {
    int signal_norm, symmetric_norm, clip_norm;
    float max_norm, min_level_db, ref_level_db;
    const float* scaler_mean;
    const float* scaler_scale;
} b200tts_audio_norm;
int b200tts_vocoder_input_len(int T, float scale_factor, int padding);
int b200tts_vocoder_input(const float* x, long long x_batch_stride, int x_channel_stride, int x_time_stride, int B, int C,
                          int T, const b200tts_audio_norm* denormalize, const b200tts_audio_norm* normalize,
                          float scale_factor, int padding, float* y, int y_pitch, void* stream);
int b200tts_absmax(const float* x, long long n, uint32_t* peak_bits, void* stream);
int b200tts_to_int16(const float* x, long long n, const uint32_t* peak_bits, int16_t* out, void* stream);

/* ---- residual-coupling flow, reverse direction ------------------------------------------------
 * Replaces ResidualCouplingBlocks.forward(reverse=True), TTS/tts/layers/vits/networks.py:214-232
 * (blocks :138-166, WaveNet TTS/tts/layers/generic/wavenet.py:94-115) as called at vits.py:1156.
 * weights per flow n = 0..num_flows-1 (host, PyTorch layouts, weight norm folded):
 *   pre.w [H, C/2, 1], pre.b
 *   enc.cond_layer.w [2*H*L, cond, 1], enc.cond_layer.b            (only if cond_channels > 0)
 *   for each WN layer i: enc.in_layers[i].w [2H,H,k], .b, enc.res_skip_layers[i].w [2H or H,H,1], .b
 *   post.w [C/2, H, 1], post.b
 * z [B,C,T] is transformed IN PLACE; mask [B,T] (1/0 floats, the reference's y_mask); g [B,cond] or NULL.
 */
typedef struct {
    int channels;
    int hidden_channels;
    int kernel_size;
    int dilation_rate;
    int num_layers;
    int num_flows;
    int cond_channels;
} b200tts_flow_config;

typedef struct b200tts_flow b200tts_flow;
int b200tts_flow_create(const b200tts_flow_config* cfg, const float* const* weights, int num_weights,
                        b200tts_flow** out);
/* same weights, packed for the forward direction (networks.py:223-227; voice conversion, vits.py:1226):
 * run it with b200tts_flow_reverse() -- the handle remembers its direction */
int b200tts_flow_create_forward(const b200tts_flow_config* cfg, const float* const* weights, int num_weights,
                                b200tts_flow** out);
void b200tts_flow_destroy(b200tts_flow* h);
size_t b200tts_flow_workspace_bytes(const b200tts_flow* h, int B, int T);
int b200tts_flow_reverse(const b200tts_flow* h, float* z, const float* mask, const float* g, int B, int T,
                         void* workspace, size_t workspace_bytes, void* stream);
/* Same with frame_lengths (device int32 [B], = the row sums of mask): rows are neither computed nor read past their
 * length.  Everything in the flow is re-masked, so frames below frame_lengths[b] are bit-identical to the dense call;
 * beyond a row's end z keeps its input values (the dense call writes zeros there): mask z afterwards. */
int b200tts_flow_reverse_ragged(const b200tts_flow* h, float* z, const float* mask, const float* g,
                                const int32_t* frame_lengths, int B, int T, void* workspace, size_t workspace_bytes,
                                void* stream);

/* ---- latent upsampling (VitsArgs.encoder_sample_rate) -----------------------------------------
 * Replaces torch.nn.functional.interpolate(z, scale_factor=[f], mode="linear") in Vits.upsampling_z,
 * TTS/tts/models/vits.py:944-959.  x [rows, Tin] -> y [rows, Tout], Tout = floor(Tin * f) chosen by the caller.
 */
int b200tts_upsample_linear(const float* x, int rows, int Tin, float scale_factor, float* y, int Tout, void* stream);

/* ---- posterior encoder (training / voice conversion) ----------------------------------------
 * Replaces PosteriorEncoder.forward, TTS/tts/layers/vits/networks.py:275-288.
 * weights: pre.w [H,Cin,1], pre.b, [enc.cond_layer.w, .b], per WN layer enc.in_layers[i].w,.b, enc.res_skip_layers[i].w,.b,
 *          proj.w [2*out,H,1], proj.b.
 * x [B,Cin,T] (linear spectrogram); mask [B,T]; g [B,cond] or NULL; noise [B,out,T] = the randn_like(mean) draw of :287.
 * outputs: z [B,out,T] = (mean + noise*exp(log_scale))*mask; stats [B,2*out,T] = [mean | log_scale] (masked).
 */
typedef struct {
    int in_channels;
    int out_channels;
    int hidden_channels;
    int kernel_size;
    int dilation_rate;
    int num_layers;
    int cond_channels;
} b200tts_posterior_config;
typedef struct b200tts_posterior b200tts_posterior;
int b200tts_posterior_create(const b200tts_posterior_config* cfg, const float* const* weights, int num_weights,
                             b200tts_posterior** out);
void b200tts_posterior_destroy(b200tts_posterior* h);
size_t b200tts_posterior_workspace_bytes(const b200tts_posterior* h, int B, int T);
int b200tts_posterior_forward(const b200tts_posterior* h, const float* x, const float* mask, const float* g,
                              const float* noise, int B, int T, float* z, float* stats, void* workspace,
                              size_t workspace_bytes, void* stream);

/* ---- deterministic duration predictor (VitsArgs.use_sdp = False) ----------------------------
 * Replaces DurationPredictor.forward, TTS/tts/layers/glow_tts/duration_predictor.py:44-69.
 * weights: conv_1.w [F,Cin,k], .b, norm_1.gamma [F], .beta, conv_2.w [F,F,k], .b, norm_2.gamma, .beta, proj.w [1,F,1], .b,
 *          [cond.w [Cin,cond,1], .b], [cond_lang.w [Cin,L,1], .b]          (Cin = in_channels + language_emb_dim)
 * x [B,Cin,T]; mask [B,T]; g [B,cond] / lang_emb [B,L] or NULL -> log-durations [B,T].
 */
typedef struct {
    int in_channels;
    int hidden_channels;
    int kernel_size;
    int cond_channels;
    int language_emb_dim;
} b200tts_duration_predictor_config;
typedef struct b200tts_duration_predictor b200tts_duration_predictor;
int b200tts_duration_predictor_create(const b200tts_duration_predictor_config* cfg, const float* const* weights,
                                      int num_weights, b200tts_duration_predictor** out);
void b200tts_duration_predictor_destroy(b200tts_duration_predictor* h);
size_t b200tts_duration_predictor_workspace_bytes(const b200tts_duration_predictor* h, int B, int T);
int b200tts_duration_predictor_forward(const b200tts_duration_predictor* h, const float* x, const float* mask,
                                       const float* g, const float* lang_emb, int B, int T, float* logw,
                                       void* workspace, size_t workspace_bytes, void* stream);

/* ---- text encoder ----------------------------------------------------------------------------
 * Replaces TextEncoder.forward, TTS/tts/layers/vits/networks.py:80-100 (RelativePositionTransformer
 * TTS/tts/layers/glow_tts/transformer.py:411-432, layer_norm_type "2", heads_share=True).
 * weights (host): emb.weight [n_vocab, hidden];
 *   per layer l: attn.emb_rel_k [1,2w+1,d], attn.emb_rel_v, conv_q.w,.b, conv_k.w,.b, conv_v.w,.b, conv_o.w,.b,
 *                norm_layers_1.gamma,.beta, ffn.conv_1.w,.b, ffn.conv_2.w,.b, norm_layers_2.gamma,.beta
 *   proj.w [2*out, C, 1], proj.b                      (C = hidden_channels + language_emb_dim)
 * tokens int64 [B,T]; lengths int64 [B]; lang_emb [B, language_emb_dim] or NULL.
 * outputs: x [B,C,T]; stats [B,2*out,T] (m_p = rows [0,out), logs_p = rows [out,2*out)); x_mask [B,T].
 */
typedef struct {
    int n_vocab;
    int out_channels;
    int hidden_channels;
    int hidden_channels_ffn;
    int num_heads;
    int num_layers;
    int kernel_size;
    int rel_attn_window_size;
    int language_emb_dim;
} b200tts_text_encoder_config;

typedef struct b200tts_text_encoder b200tts_text_encoder;
int b200tts_text_encoder_create(const b200tts_text_encoder_config* cfg, const float* const* weights,
                                int num_weights, b200tts_text_encoder** out);
void b200tts_text_encoder_destroy(b200tts_text_encoder* h);
size_t b200tts_text_encoder_workspace_bytes(const b200tts_text_encoder* h, int B, int T);
int b200tts_text_encoder_forward(const b200tts_text_encoder* h, const int64_t* tokens, const int64_t* lengths,
                                 const float* lang_emb, int B, int T, float* x, float* stats, float* x_mask,
                                 void* workspace, size_t workspace_bytes, void* stream);

/* ---- stochastic duration predictor, reverse ---------------------------------------------------
 * Replaces StochasticDurationPredictor.forward(reverse=True),
 * TTS/tts/layers/vits/stochastic_duration_predictor.py:222-239,285-294 (+ transforms.py spline inverse).
 * weights (host): pre.w [H,in,1], pre.b; [cond.w, cond.b]; [cond_lang.w, cond_lang.b];
 *   convs: 3 x (convs_sep.w [H,1,k], .b, convs_1x1.w [H,H,1], .b, norms_1.gamma,.beta, norms_2.gamma,.beta);
 *   proj.w [H,H,1], proj.b; flows.0.translation [2], flows.0.log_scale [2];
 *   for f = 1..num_flows: flows.f.pre.w [H,1,1], .b, flows.f.convs (3 x 8 as above), flows.f.proj.w [3*nb-1,H,1], .b
 * x [B,in,T]; mask [B,T]; noise [B,2,T] = the standard-normal draw of :287 (made by the caller so
 * that results are reproducible against the reference); g [B,cond] / lang_emb [B,L] or NULL.
 * logw [B,T].  err_flag: device int set to 1 if the spline discriminant goes negative (the reference
 * asserts, transforms.py:168); may be NULL.
 */
typedef struct {
    int in_channels;
    int hidden_channels;
    int kernel_size;
    int num_flows;
    int cond_channels;
    int language_emb_dim;
    int num_bins;
    float tail_bound;
} b200tts_sdp_config;

typedef struct b200tts_sdp b200tts_sdp;
int b200tts_sdp_create(const b200tts_sdp_config* cfg, const float* const* weights, int num_weights,
                       b200tts_sdp** out);
void b200tts_sdp_destroy(b200tts_sdp* h);
size_t b200tts_sdp_workspace_bytes(const b200tts_sdp* h, int B, int T);
int b200tts_sdp_reverse(const b200tts_sdp* h, const float* x, const float* mask, const float* noise, const float* g,
                        const float* lang_emb, float noise_scale, int B, int T, float* logw, int32_t* err_flag,
                        void* workspace, size_t workspace_bytes, void* stream);

/* ---- durations -> path -> expanded prior ------------------------------------------------------
 * Replaces the glue at TTS/tts/models/vits.py:1140-1155 (generate_path: TTS/tts/utils/helpers.py:154-169).
 * b200tts_durations : w_ceil [B,T] = ceil(exp(logw) * x_mask * length_scale); cum [B,T] = cumsum(w_ceil);
 *                     y_lengths int64 [B] = max(1, sum(w_ceil)); meta int64 [2] (or NULL) = {max_b y_lengths,
 *                     *err_flag (the duration predictor's spline flag, may be NULL -> 0)}: the one host read of
 *                     Vits.inference (sequence_mask(y_lengths, None), helpers.py:53-54) fetches both.
 * b200tts_expand_prior (after the caller has read max(y_lengths) = Ty): attn [B,Tx,Ty] one-hot (or NULL),
 *   m_p / logs_p / z_p [B,C,Ty] with z_p = m_p + noise * exp(logs_p) * noise_scale, y_mask [B,Ty] (or NULL);
 *   stats is the text encoder's [B,2C,Tx]; noise [B,C,Ty] is the randn_like(m_p) draw of vits.py:1155.
 */
int b200tts_durations(const float* logw, const float* x_mask, float length_scale, int B, int T, float* w_ceil,
                      float* cum, int64_t* y_lengths, const int32_t* err_flag, int64_t* meta, void* stream);
int b200tts_expand_prior(const float* cum, const float* x_mask, const int64_t* y_lengths, const float* stats,
                         const float* noise, float noise_scale, int B, int Tx, int Ty, int C, float* attn,
                         float* m_p, float* logs_p, float* z_p, float* y_mask, void* stream);

/* ---- STFT magnitude / mel front end ----------------------------------------------------------
 * Replaces wav_to_spec / spec_to_mel / wav_to_mel, TTS/tts/models/vits.py:96-208, and TorchSTFT.__call__,
 * TTS/utils/audio/torch_transforms.py:104-145.
 * create: window [n_fft] (host; the analysis window already zero-padded to n_fft), mel_basis [n_mels, n_fft/2+1]
 *         (host, e.g. librosa.filters.mel) or NULL.  n_fft must be a power of two.
 * magnitude: wav [B,T] -> spec [B, n_fft/2+1, n_frames].  The signal is reflect-padded by pad1 samples, then by
 *   pad2 samples (both each side; 0 = none), then framed with hop (no centering of its own):
 *     wav_to_spec  : pad1 = (n_fft-hop)/2, pad2 = 0,        mode 0: sqrt(re^2+im^2+1e-6)
 *     TorchSTFT    : pad1 = pad_wav ? (n_fft-hop)/2 : 0, pad2 = n_fft/2 (center=True), mode 1: sqrt(max(.,1e-8))
 *   power != 1 raises the magnitude to that power (TorchSTFT.power).
 * mel_project: mel [B,n_mels,n_frames] = basis @ spec, followed by log(max(., log_clamp)) when log_clamp > 0.
 */
typedef struct b200tts_stft b200tts_stft;
int b200tts_stft_create(int n_fft, int hop_length, const float* window, const float* mel_basis, int n_mels,
                        b200tts_stft** out);
void b200tts_stft_destroy(b200tts_stft* h);
int b200tts_stft_magnitude(const b200tts_stft* h, const float* wav, int B, int T, int pad1, int pad2, int mode,
                           float power, float* spec, int n_frames, void* stream);
int b200tts_stft_mel_project(const b200tts_stft* h, const float* spec, int B, int n_frames, float log_clamp,
                             float* mel, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* TTS_B200_H */
