// extern "C" surface of libtts_b200.so -- see include/tts_b200.h for the contract.
#include <new>

#include "engines.cuh"

using namespace b200tts;

struct b200tts_hifigan { Hifigan impl; };
struct b200tts_flow { Flow impl; };
struct b200tts_text_encoder { TextEncoder impl; };
struct b200tts_sdp { SDP impl; };
struct b200tts_stft { Stft impl; };
struct b200tts_posterior { PosteriorEnc impl; };
struct b200tts_duration_predictor { DurPred impl; };

extern "C" {

const char* b200tts_last_error(void) { return last_error(); }
unsigned long long b200tts_launch_count(void) { return g_launch_count; }
int b200tts_version(void) { return 101; }
int b200tts_debug_tc_error(void) { return conv_tc_error_flag(); }
void b200tts_debug_dispatch_begin(void) { dispatch_begin(); }
int b200tts_debug_dispatch_end(int32_t* ids, int cap) { return dispatch_end(ids, cap); }

struct b200tts_conv1d { ConvLayer L; b200tts_conv1d_config c; ~b200tts_conv1d() { free_conv(L); } };

static bool known_precision(int p) { return p == B200TTS_PRECISION_FP32 || p == B200TTS_PRECISION_TF32; }

int b200tts_conv1d_create(const b200tts_conv1d_config* cfg, const float* weight, const float* bias, int allow_tensor_cores,
                          b200tts_conv1d** out) {
    return b200tts_conv1d_create_ex(cfg, weight, bias, allow_tensor_cores, B200TTS_PRECISION_FP32, out);
}
int b200tts_conv1d_create_ex(const b200tts_conv1d_config* cfg, const float* weight, const float* bias, int allow_tensor_cores,
                             int precision, b200tts_conv1d** out) {
    if (!cfg || !weight || !out) { set_error("conv1d_create: null argument"); return 1; }
    *out = nullptr;
    if (!known_precision(precision)) { set_error("conv1d_create: unknown precision %d", precision); return 1; }
    const int tp = precision == B200TTS_PRECISION_TF32 ? 1 : 3;
    b200tts_conv1d* h = new (std::nothrow) b200tts_conv1d();
    if (!h) { set_error("conv1d_create: out of host memory"); return 1; }
    h->c = *cfg;
    int rc = cfg->transposed
                 ? pack_conv_transpose(h->L, weight, bias, cfg->in_channels, cfg->out_channels, cfg->kernel_size,
                                       cfg->stride, cfg->padding, tp)
                 : pack_conv(h->L, weight, bias, cfg->out_channels, cfg->in_channels, cfg->kernel_size, cfg->dilation,
                             cfg->padding, 0, nullptr, nullptr, tp);
    if (rc) { delete h; return rc; }
    h->L.allow_tc = allow_tensor_cores != 0;
    *out = h;
    return 0;
}
void b200tts_conv1d_destroy(b200tts_conv1d* h) { delete h; }
int b200tts_conv1d_out_len(const b200tts_conv1d* h, int T) {
    if (!h) return 0;
    if (h->c.transposed) return conv_transpose_out_len(h->L, T);
    return T + 2 * h->c.padding - h->c.dilation * (h->c.kernel_size - 1);
}
int b200tts_conv1d_forward(const b200tts_conv1d* h, const float* x, int B, int T, float in_slope, const float* residual,
                           float scale, int accumulate, float post_div, float* y, void* stream) {
    if (!h) { set_error("conv1d_forward: null handle"); return 1; }
    const int Tout = b200tts_conv1d_out_len(h, T);
    ConvIO io;
    io.x = x; io.x_bs = (long long)h->c.in_channels * T; io.x_cs = T; io.Tin = T; io.in_slope = in_slope;
    io.y = y; io.y_bs = (long long)h->c.out_channels * Tout; io.y_cs = Tout; io.Tout = Tout; io.B = B;
    if (residual) { io.res = residual; io.res_bs = io.y_bs; io.res_cs = Tout; }
    io.scale = scale; io.post_div = post_div;
    if (accumulate) io.flags |= EPI_ACCUM;
    return launch_conv(h->L, io, (cudaStream_t)stream);
}

size_t b200tts_mas_workspace_bytes(int B, int Tx, int Ty) { return mas_workspace_bytes(B, Tx, Ty); }

int b200tts_mas(const float* value, const float* mask, const int32_t* t_x, const int32_t* t_y, int B, int Tx,
                int Ty, void* path, int path_is_f32, void* workspace, size_t workspace_bytes, void* stream) {
    return mas_forward(value, mask, t_x, t_y, B, Tx, Ty, path, path_is_f32, workspace, workspace_bytes,
                       (cudaStream_t)stream);
}

size_t b200tts_mas_from_stats_workspace_bytes(int B, int Tx, int Ty) { return mas_from_stats_workspace_bytes(B, Tx, Ty); }
int b200tts_mas_from_stats(const float* z_p, const float* m_p, const float* logs_p, const int32_t* t_x, const int32_t* t_y,
                           int B, int C, int Tx, int Ty, void* path, int path_is_f32, float* logp_out, void* workspace,
                           size_t workspace_bytes, void* stream) {
    return mas_from_stats(z_p, m_p, logs_p, t_x, t_y, B, C, Tx, Ty, path, path_is_f32, logp_out, workspace, workspace_bytes,
                          (cudaStream_t)stream);
}

int b200tts_hifigan_create(const b200tts_hifigan_config* cfg, const float* const* weights, int num_weights,
                           b200tts_hifigan** out) {
    return b200tts_hifigan_create_ex(cfg, weights, num_weights, B200TTS_PRECISION_FP32, out);
}
int b200tts_hifigan_create_ex(const b200tts_hifigan_config* cfg, const float* const* weights, int num_weights, int precision,
                              b200tts_hifigan** out) {
    if (!cfg || !weights || !out) { set_error("hifigan_create: null argument"); return 1; }
    *out = nullptr;
    if (!known_precision(precision)) { set_error("hifigan_create: unknown precision %d", precision); return 1; }
    b200tts_hifigan* h = new (std::nothrow) b200tts_hifigan();
    if (!h) { set_error("hifigan_create: out of host memory"); return 1; }
    int rc = h->impl.init(*cfg, weights, num_weights, precision);
    if (rc) { delete h; return rc; }
    *out = h;
    return 0;
}
int b200tts_hifigan_precision(const b200tts_hifigan* h) { return h ? h->impl.precision : -1; }
void b200tts_hifigan_destroy(b200tts_hifigan* h) { delete h; }
size_t b200tts_hifigan_workspace_bytes(const b200tts_hifigan* h, int B, int T) {
    return h ? h->impl.workspace_bytes(B, T) : 0;
}
int b200tts_hifigan_out_len(const b200tts_hifigan* h, int T) { return h ? h->impl.out_len(T) : 0; }
int b200tts_hifigan_forward(const b200tts_hifigan* h, const float* x, const float* g, int B, int T, float* wav,
                            void* workspace, size_t workspace_bytes, void* stream) {
    if (!h) { set_error("hifigan_forward: null handle"); return 1; }
    return h->impl.forward(x, g, B, T, wav, workspace, workspace_bytes, (cudaStream_t)stream);
}

int b200tts_hifigan_forward_ex(const b200tts_hifigan* h, const float* x, const float* g, int B, int T, float* wav,
                               const int32_t* frame_lengths, uint32_t* peak_bits, void* workspace, size_t workspace_bytes,
                               void* stream) {
    if (!h) { set_error("hifigan_forward_ex: null handle"); return 1; }
    return h->impl.forward(x, g, B, T, wav, workspace, workspace_bytes, (cudaStream_t)stream, peak_bits, frame_lengths);
}
int b200tts_hifigan_margin_frames(const b200tts_hifigan* h) {   // frames past a row's end the ragged schedule still computes
    return h ? h->impl.need_P : 0;
}

int b200tts_vocoder_input_len(int T, float scale_factor, int padding) { return vocoder_input_len(T, scale_factor, padding); }
int b200tts_vocoder_input(const float* x, long long x_batch_stride, int x_channel_stride, int x_time_stride, int B, int C,
                          int T, const b200tts_audio_norm* denormalize, const b200tts_audio_norm* normalize,
                          float scale_factor, int padding, float* y, int y_pitch, void* stream) {
    return launch_vocoder_input(x, x_batch_stride, x_channel_stride, x_time_stride, B, C, T, denormalize, normalize,
                                scale_factor, padding, y, y_pitch, (cudaStream_t)stream);
}
int b200tts_absmax(const float* x, long long n, uint32_t* peak_bits, void* stream) {
    return launch_absmax(x, n, peak_bits, (cudaStream_t)stream);
}
int b200tts_to_int16(const float* x, long long n, const uint32_t* peak_bits, int16_t* out, void* stream) {
    return launch_to_int16(x, n, peak_bits, out, (cudaStream_t)stream);
}

int b200tts_flow_create(const b200tts_flow_config* cfg, const float* const* weights, int num_weights,
                        b200tts_flow** out) {
    if (!cfg || !weights || !out) { set_error("flow_create: null argument"); return 1; }
    *out = nullptr;
    b200tts_flow* h = new (std::nothrow) b200tts_flow();
    if (!h) { set_error("flow_create: out of host memory"); return 1; }
    int rc = h->impl.init(*cfg, weights, num_weights);
    if (rc) { delete h; return rc; }
    *out = h;
    return 0;
}
int b200tts_flow_create_forward(const b200tts_flow_config* cfg, const float* const* weights, int num_weights,
                                b200tts_flow** out) {
    if (!cfg || !weights || !out) { set_error("flow_create_forward: null argument"); return 1; }
    *out = nullptr;
    b200tts_flow* h = new (std::nothrow) b200tts_flow();
    if (!h) { set_error("flow_create_forward: out of host memory"); return 1; }
    int rc = h->impl.init(*cfg, weights, num_weights, 1);
    if (rc) { delete h; return rc; }
    *out = h;
    return 0;
}
void b200tts_flow_destroy(b200tts_flow* h) { delete h; }
size_t b200tts_flow_workspace_bytes(const b200tts_flow* h, int B, int T) {
    return h ? h->impl.workspace_bytes(B, T) : 0;
}
int b200tts_flow_reverse(const b200tts_flow* h, float* z, const float* mask, const float* g, int B, int T,
                         void* workspace, size_t workspace_bytes, void* stream) {
    if (!h) { set_error("flow_reverse: null handle"); return 1; }
    return h->impl.reverse(z, mask, g, B, T, workspace, workspace_bytes, (cudaStream_t)stream);
}
int b200tts_flow_reverse_ragged(const b200tts_flow* h, float* z, const float* mask, const float* g,
                                const int32_t* frame_lengths, int B, int T, void* workspace, size_t workspace_bytes,
                                void* stream) {
    if (!h) { set_error("flow_reverse_ragged: null handle"); return 1; }
    return h->impl.reverse(z, mask, g, B, T, workspace, workspace_bytes, (cudaStream_t)stream, frame_lengths);
}

int b200tts_text_encoder_create(const b200tts_text_encoder_config* cfg, const float* const* weights,
                                int num_weights, b200tts_text_encoder** out) {
    if (!cfg || !weights || !out) { set_error("text_encoder_create: null argument"); return 1; }
    *out = nullptr;
    b200tts_text_encoder* h = new (std::nothrow) b200tts_text_encoder();
    if (!h) { set_error("text_encoder_create: out of host memory"); return 1; }
    int rc = h->impl.init(*cfg, weights, num_weights);
    if (rc) { delete h; return rc; }
    *out = h;
    return 0;
}
void b200tts_text_encoder_destroy(b200tts_text_encoder* h) { delete h; }
size_t b200tts_text_encoder_workspace_bytes(const b200tts_text_encoder* h, int B, int T) {
    return h ? h->impl.workspace_bytes(B, T) : 0;
}
int b200tts_text_encoder_forward(const b200tts_text_encoder* h, const int64_t* tokens, const int64_t* lengths,
                                 const float* lang_emb, int B, int T, float* x, float* stats, float* x_mask,
                                 void* workspace, size_t workspace_bytes, void* stream) {
    if (!h) { set_error("text_encoder_forward: null handle"); return 1; }
    return h->impl.forward((const long long*)tokens, (const long long*)lengths, lang_emb, B, T, x, stats, x_mask,
                           workspace, workspace_bytes, (cudaStream_t)stream);
}

int b200tts_sdp_create(const b200tts_sdp_config* cfg, const float* const* weights, int num_weights,
                       b200tts_sdp** out) {
    if (!cfg || !weights || !out) { set_error("sdp_create: null argument"); return 1; }
    *out = nullptr;
    b200tts_sdp* h = new (std::nothrow) b200tts_sdp();
    if (!h) { set_error("sdp_create: out of host memory"); return 1; }
    int rc = h->impl.init(*cfg, weights, num_weights);
    if (rc) { delete h; return rc; }
    *out = h;
    return 0;
}
void b200tts_sdp_destroy(b200tts_sdp* h) { delete h; }
size_t b200tts_sdp_workspace_bytes(const b200tts_sdp* h, int B, int T) { return h ? h->impl.workspace_bytes(B, T) : 0; }
int b200tts_sdp_reverse(const b200tts_sdp* h, const float* x, const float* mask, const float* noise, const float* g,
                        const float* lang_emb, float noise_scale, int B, int T, float* logw, int32_t* err_flag,
                        void* workspace, size_t workspace_bytes, void* stream) {
    if (!h) { set_error("sdp_reverse: null handle"); return 1; }
    return h->impl.reverse(x, mask, noise, g, lang_emb, noise_scale, B, T, logw, err_flag, workspace, workspace_bytes,
                           (cudaStream_t)stream);
}

int b200tts_durations(const float* logw, const float* x_mask, float length_scale, int B, int T, float* w_ceil,
                      float* cum, int64_t* y_lengths, const int32_t* err_flag, int64_t* meta, void* stream) {
    return launch_durations(logw, x_mask, length_scale, B, T, w_ceil, cum, (long long*)y_lengths, err_flag,
                            (long long*)meta, (cudaStream_t)stream);
}
int b200tts_expand_prior(const float* cum, const float* x_mask, const int64_t* y_lengths, const float* stats,
                         const float* noise, float noise_scale, int B, int Tx, int Ty, int C, float* attn,
                         float* m_p, float* logs_p, float* z_p, float* y_mask, void* stream) {
    return launch_expand_prior(cum, x_mask, (const long long*)y_lengths, stats, noise, noise_scale, B, Tx, Ty, C, attn,
                               m_p, logs_p, z_p, y_mask, (cudaStream_t)stream);
}

int b200tts_upsample_linear(const float* x, int rows, int Tin, float scale_factor, float* y, int Tout, void* stream) {
    return launch_upsample_linear(x, rows, Tin, scale_factor, y, Tout, (cudaStream_t)stream);
}

int b200tts_stft_create(int n_fft, int hop_length, const float* window, const float* mel_basis, int n_mels,
                        b200tts_stft** out) {
    if (!out) { set_error("stft_create: null argument"); return 1; }
    *out = nullptr;
    b200tts_stft* h = new (std::nothrow) b200tts_stft();
    if (!h) { set_error("stft_create: out of host memory"); return 1; }
    int rc = h->impl.init(n_fft, hop_length, window, mel_basis, n_mels);
    if (rc) { delete h; return rc; }
    *out = h;
    return 0;
}
void b200tts_stft_destroy(b200tts_stft* h) { delete h; }
int b200tts_stft_magnitude(const b200tts_stft* h, const float* wav, int B, int T, int pad1, int pad2, int mode,
                           float power, float* spec, int n_frames, void* stream) {
    if (!h) { set_error("stft_magnitude: null handle"); return 1; }
    return h->impl.magnitude(wav, B, T, pad1, pad2, mode, power, spec, n_frames, (cudaStream_t)stream);
}
int b200tts_stft_mel_project(const b200tts_stft* h, const float* spec, int B, int n_frames, float log_clamp,
                             float* mel, void* stream) {
    if (!h) { set_error("stft_mel_project: null handle"); return 1; }
    return h->impl.mel_project(spec, B, n_frames, log_clamp, mel, (cudaStream_t)stream);
}

#define B200_HANDLE_API(NAME, TYPE, CFG)                                                                        \
    int b200tts_##NAME##_create(const CFG* cfg, const float* const* weights, int num_weights, TYPE** out) {       \
        if (!cfg || !weights || !out) { set_error(#NAME "_create: null argument"); return 1; }                   \
        *out = nullptr;                                                                                          \
        TYPE* h = new (std::nothrow) TYPE();                                                                     \
        if (!h) { set_error(#NAME "_create: out of host memory"); return 1; }                                    \
        int rc = h->impl.init(*cfg, weights, num_weights);                                                       \
        if (rc) { delete h; return rc; }                                                                         \
        *out = h;                                                                                                \
        return 0;                                                                                                \
    }                                                                                                            \
    void b200tts_##NAME##_destroy(TYPE* h) { delete h; }                                                         \
    size_t b200tts_##NAME##_workspace_bytes(const TYPE* h, int B, int T) { return h ? h->impl.workspace_bytes(B, T) : 0; }

B200_HANDLE_API(posterior, b200tts_posterior, b200tts_posterior_config)
B200_HANDLE_API(duration_predictor, b200tts_duration_predictor, b200tts_duration_predictor_config)

int b200tts_posterior_forward(const b200tts_posterior* h, const float* x, const float* mask, const float* g,
                              const float* noise, int B, int T, float* z, float* stats, void* workspace,
                              size_t workspace_bytes, void* stream) {
    if (!h) { set_error("posterior_forward: null handle"); return 1; }
    return h->impl.forward(x, mask, g, noise, B, T, z, stats, workspace, workspace_bytes, (cudaStream_t)stream);
}
int b200tts_duration_predictor_forward(const b200tts_duration_predictor* h, const float* x, const float* mask,
                                       const float* g, const float* lang_emb, int B, int T, float* logw,
                                       void* workspace, size_t workspace_bytes, void* stream) {
    if (!h) { set_error("duration_predictor_forward: null handle"); return 1; }
    return h->impl.forward(x, mask, g, lang_emb, B, T, logw, workspace, workspace_bytes, (cudaStream_t)stream);
}

}  // extern "C"
