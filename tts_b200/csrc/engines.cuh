// Engine handles behind the C ABI (include/tts_b200.h).  Immutable after init(): safe to share
// across streams/threads; all scratch comes from the caller's workspace.
#pragma once
#include <algorithm>
#include <string.h>

#include "../../include/tts_b200.h"
#include "common.cuh"

namespace b200tts {

struct Hifigan {
    b200tts_hifigan_config c;
    ConvLayer conv_pre, cond, conv_post;
    std::vector<ConvLayer> ups;
    std::vector<std::vector<ConvLayer>> rb_c1, rb_c2;
    int precision = B200TTS_PRECISION_FP32;   // B200TTS_PRECISION_*: how the tensor-core layers were packed
    ~Hifigan();
    int init(const b200tts_hifigan_config& cfg, const float* const* w, int nw, int precision = B200TTS_PRECISION_FP32);
    void stage_dims(int T, std::vector<int>& C, std::vector<int>& L) const;
    size_t workspace_bytes(int B, int T) const;
    int out_len(int T) const;
    // peak_bits (nullable): device word that conv_post's store folds max|wav| into (atomicMax on the float's bits; the
    // caller zeroes it) -- the first half of save_wav's peak normalisation without another pass over the waveform
    // lens (nullable, device int32 [B]): valid frames per row.  With it, padded frames are neither computed nor read:
    // every launch stops `need` samples past a row's end, where `need` is the receptive field of the layers that still
    // follow (worked out in init()), so all samples below lens[b] * prod(upsample_factors) are bit-identical to the dense
    // call; the rest of the row is zero.
    int forward(const float* x, const float* g, int B, int T, float* wav, void* ws, size_t ws_bytes,
                cudaStream_t st, unsigned* peak_bits = nullptr, const int* lens = nullptr) const;
    // per-launch exactness margins (samples at the tensor's own rate), see init()
    int need_P = 0;
    std::vector<int> need_OUT, need_U, need_q_ups, rate;
    std::vector<std::vector<int>> need_T1, need_X;
    void plan_margins();
};

struct WaveNet {
    int H = 0, K = 0, L = 0, cond_ch = 0;
    ConvLayer cond;
    std::vector<ConvLayer> in_layers, res_skip;
    ~WaveNet();
    int init(int hidden, int kernel_size, int dilation_rate, int num_layers, int cond_channels,
             const float* const* w, int* consumed);
    size_t scratch_floats(int B, int T) const;
    int forward(float* h, float* out, const float* mask, const float* g, int B, int T, float* acts, float* condv,
                cudaStream_t st, const int* lens = nullptr) const;
};

struct Flow {
    struct Block { ConvLayer pre, post; WaveNet wn; bool odd = false; };
    b200tts_flow_config c;
    bool fwd = false;
    std::vector<Block*> blocks;
    ~Flow();
    int init(const b200tts_flow_config& cfg, const float* const* w, int nw, int forward_direction = 0);
    size_t workspace_bytes(int B, int T) const;
    // lens (nullable, device int32 [B]): frames per row; rows are neither computed nor read past their length (every
    // tensor in the flow is re-masked, so the frames below lens[b] are bit-identical to the dense call; z keeps its
    // input values beyond a row's end instead of the zeros the masking would write -- callers mask z afterwards)
    int reverse(float* z, const float* mask, const float* g, int B, int T, void* ws, size_t ws_bytes,
                cudaStream_t st, const int* lens = nullptr) const;
};

struct PosteriorEnc {
    b200tts_posterior_config c;
    ConvLayer pre, proj;
    WaveNet wn;
    ~PosteriorEnc();
    int init(const b200tts_posterior_config& cfg, const float* const* w, int nw);
    size_t workspace_bytes(int B, int T) const;
    int forward(const float* x, const float* mask, const float* g, const float* noise, int B, int T, float* z,
                float* stats, void* ws, size_t ws_bytes, cudaStream_t st) const;
};

struct DurPred {
    b200tts_duration_predictor_config c;
    ConvLayer conv1, conv2, proj, cond, cond_lang;
    float *g1 = nullptr, *b1 = nullptr, *g2 = nullptr, *b2 = nullptr;
    ~DurPred();
    int init(const b200tts_duration_predictor_config& cfg, const float* const* w, int nw);
    size_t workspace_bytes(int B, int T) const;
    int forward(const float* x, const float* mask, const float* g, const float* lang_emb, int B, int T, float* logw,
                void* ws, size_t ws_bytes, cudaStream_t st) const;
};

int launch_upsample_linear(const float* x, int rows, int Tin, float scale_factor, float* y, int Tout, cudaStream_t st);
int launch_add_layernorm(const float* x, const float* y, const float* gamma, const float* beta, const float* mask,
                         float* out, int B, int C, int T, float eps, cudaStream_t st);

struct TextEncoder {
    struct Layer {
        ConvLayer qkv, o, ffn1, ffn2;
        float *rel_k = nullptr, *rel_v = nullptr, *ln1_g = nullptr, *ln1_b = nullptr, *ln2_g = nullptr, *ln2_b = nullptr;
    };
    b200tts_text_encoder_config c;
    int C = 0, d = 0;
    float* emb = nullptr;
    std::vector<Layer*> layers;
    ConvLayer proj;
    ~TextEncoder();
    int init(const b200tts_text_encoder_config& cfg, const float* const* w, int nw);
    size_t workspace_bytes(int B, int T) const;
    int forward(const long long* tokens, const long long* lengths, const float* lang_emb, int B, int T, float* x,
                float* stats, float* x_mask, void* ws, size_t ws_bytes, cudaStream_t st) const;
};

struct DDSConv {
    int C = 0, K = 0, L = 0;
    std::vector<ConvLayer> conv1x1;
    std::vector<float*> sep_w, sep_b, g1, b1, g2, b2, dev;
    ~DDSConv();
    int init(int channels, int kernel_size, int num_layers, const float* const* w, int* consumed);
    int forward(float* x, const float* mask, int B, int T, float* y1, float* y2, cudaStream_t st) const;
};

struct SDP {
    struct CFlow { float *pre_w = nullptr, *pre_b = nullptr; DDSConv convs; ConvLayer proj; };
    b200tts_sdp_config c;
    ConvLayer pre, cond, cond_lang, proj;
    DDSConv convs;
    float *ea_t = nullptr, *ea_ls = nullptr;
    std::vector<CFlow*> flows;
    ~SDP();
    int init(const b200tts_sdp_config& cfg, const float* const* w, int nw);
    size_t workspace_bytes(int B, int T) const;
    int reverse(const float* x, const float* mask, const float* noise, const float* g, const float* lang_emb,
                float noise_scale, int B, int T, float* logw, int* err_flag, void* ws, size_t ws_bytes,
                cudaStream_t st) const;
};

struct Stft {
    int n_fft = 0, hop = 0, log2n = 0, n_mels = 0;
    float *window = nullptr, *twiddle = nullptr;
    ConvLayer mel;
    ~Stft();
    int init(int n_fft, int hop, const float* window_host, const float* mel_basis_host, int n_mels);
    int magnitude(const float* wav, int B, int T, int pad1, int pad2, int mode, float power, float* spec, int n_frames,
                  cudaStream_t st) const;
    int mel_project(const float* spec, int B, int n_frames, float log_clamp, float* out, cudaStream_t st) const;
};

// durations -> path -> expanded prior (path.cu)
int launch_durations(const float* logw, const float* x_mask, float length_scale, int B, int T, float* w_ceil,
                     float* cum, long long* y_lengths, const int* err_flag, long long* meta, cudaStream_t st);
int launch_expand_prior(const float* cum, const float* x_mask, const long long* y_lengths, const float* stats,
                        const float* noise, float noise_scale, int B, int Tx, int Ty, int C, float* attn, float* m_p,
                        float* logs_p, float* z_p, float* y_mask, cudaStream_t st);

// vocoder hand-off (vocoder_io.cu)
int vocoder_input_len(int T, float scale_factor, int pad);
int launch_vocoder_input(const float* x, long long x_bs, int x_cs, int x_ts, int B, int C, int T,
                         const b200tts_audio_norm* denorm, const b200tts_audio_norm* norm, float scale_factor, int pad,
                         float* y, int y_pitch, cudaStream_t st);
int launch_absmax(const float* x, long long n, unsigned* peak_bits, cudaStream_t st);
int launch_to_int16(const float* x, long long n, const unsigned* peak_bits, short* out, cudaStream_t st);

// monotonic alignment search (mas.cu)
size_t mas_workspace_bytes(int B, int Tx, int Ty);
int mas_forward(const float* value, const float* mask, const int* t_x, const int* t_y, int B, int Tx, int Ty,
                void* path, int path_is_f32, void* ws, size_t ws_bytes, cudaStream_t st);
size_t mas_from_stats_workspace_bytes(int B, int Tx, int Ty);
int mas_from_stats(const float* z_p, const float* m_p, const float* logs_p, const int* t_x, const int* t_y, int B, int C,
                   int Tx, int Ty, void* path, int path_is_f32, float* logp_out, void* ws, size_t ws_bytes, cudaStream_t st);

}  // namespace b200tts
