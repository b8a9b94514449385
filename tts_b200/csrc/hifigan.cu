// HiFiGAN generator engine: launch schedule over the fused conv1d kernel.
// Reference semantics: TTS/vocoder/models/hifigan_generator.py:236-265 (HifiganGenerator.forward),
// :84-99 (ResBlock1.forward), :150-155 (ResBlock2.forward), ctor :163-234.
#include "engines.cuh"

namespace b200tts {

Hifigan::~Hifigan() {
    free_conv(conv_pre);
    free_conv(cond);
    free_conv(conv_post);
    for (auto& l : ups) free_conv(l);
    for (auto& v : rb_c1) for (auto& l : v) free_conv(l);
    for (auto& v : rb_c2) for (auto& l : v) free_conv(l);
}

// weights: host pointers, canonical order (see include/tts_b200.h)
int Hifigan::init(const b200tts_hifigan_config& cfg, const float* const* w, int nw, int prec) {
    c = cfg;
    B200_REQUIRE(prec == B200TTS_PRECISION_FP32 || prec == B200TTS_PRECISION_TF32, "hifigan: unknown precision %d", prec);
    precision = prec;
    // conv_pre, the upsamplers and the ResBlock convs are the tensor-core layers: packed for one pass in TF32 mode.
    // cond_layer and conv_post run on the FP32 kernels in either mode.
    const int tp = prec == B200TTS_PRECISION_TF32 ? 1 : 3;
    B200_REQUIRE(c.num_upsamples >= 1 && c.num_upsamples <= 8 && c.num_kernels >= 1 && c.num_kernels <= 8 &&
                     c.num_dilations >= 1 && c.num_dilations <= 8,
                 "hifigan: unsupported config");
    const int type1 = (c.resblock_type == 1);
    const int expect = 2 + (c.cond_channels > 0 ? 2 : 0) + 2 * c.num_upsamples +
                       c.num_upsamples * c.num_kernels * c.num_dilations * (type1 ? 4 : 2) + 2;
    B200_REQUIRE(nw == expect, "hifigan: expected %d weight tensors, got %d", expect, nw);
    int i = 0;
    int rc = pack_conv(conv_pre, w[i], w[i + 1], c.upsample_initial_channel, c.in_channels, 7, 1, 3, 0, nullptr, nullptr, tp);
    if (rc) return rc;
    i += 2;
    if (c.cond_channels > 0) {
        rc = pack_conv(cond, w[i], w[i + 1], c.upsample_initial_channel, c.cond_channels, 1, 1, 0);
        if (rc) return rc;
        i += 2;
    }
    ups.resize(c.num_upsamples);
    rb_c1.assign(c.num_upsamples * c.num_kernels, std::vector<ConvLayer>());
    rb_c2.assign(c.num_upsamples * c.num_kernels, std::vector<ConvLayer>());
    int ch = c.upsample_initial_channel;
    for (int s = 0; s < c.num_upsamples; ++s) {
        const int u = c.upsample_factors[s], k = c.upsample_kernel_sizes[s];
        rc = pack_conv_transpose(ups[s], w[i], w[i + 1], ch, ch / 2, k, u, (k - u) / 2, tp);
        if (rc) return rc;
        i += 2;
        ch /= 2;
        for (int j = 0; j < c.num_kernels; ++j) {
            const int rk = c.resblock_kernel_sizes[j];
            auto& v1 = rb_c1[s * c.num_kernels + j];
            auto& v2 = rb_c2[s * c.num_kernels + j];
            v1.resize(c.num_dilations);
            if (type1) v2.resize(c.num_dilations);
            for (int n = 0; n < c.num_dilations; ++n) {
                const int d = c.resblock_dilations[j][n];
                rc = pack_conv(v1[n], w[i], w[i + 1], ch, ch, rk, d, (rk * d - d) / 2, 0, nullptr, nullptr, tp);
                if (rc) return rc;
                i += 2;
                if (type1) {
                    rc = pack_conv(v2[n], w[i], w[i + 1], ch, ch, rk, 1, (rk - 1) / 2, 0, nullptr, nullptr, tp);
                    if (rc) return rc;
                    i += 2;
                }
            }
        }
    }
    rc = pack_conv(conv_post, w[i], w[i + 1], c.out_channels, ch, 7, 1, 3);
    // the MRF / pre convs carry ~97% of the FLOPs: run them on the tcgen05 kernels (3xTF32, or single pass in TF32 mode)
    conv_pre.allow_tc = true;
    for (auto& l : ups) l.allow_tc = true;
    for (auto& v : rb_c1) for (auto& l : v) l.allow_tc = true;
    for (auto& v : rb_c2) for (auto& l : v) l.allow_tc = true;
    if (rc == 0) plan_margins();
    return rc;
}

// Ragged batches: how far past a row's last valid sample must each tensor be exact so that the waveform below the
// row's end is bit-identical to the dense computation?  Walk the schedule backwards adding each layer's one-sided reach.
void Hifigan::plan_margins() {
    const int S = c.num_upsamples, nk = c.num_kernels, nd = c.num_dilations;
    const bool type1 = c.resblock_type == 1;
    need_OUT.assign(S, 0); need_U.assign(S, 0); need_q_ups.assign(S, 0); rate.assign(S, 1);
    need_T1.assign(S * nk, std::vector<int>(nd, 0));
    need_X.assign(S * nk, std::vector<int>(nd, 0));
    int r = 1;
    for (int s = 0; s < S; ++s) { r *= c.upsample_factors[s]; rate[s] = r; }
    int need_next = std::max(conv_post.pad, conv_post.K - 1 - conv_post.pad);     // what conv_post reads past a sample
    for (int s = S - 1; s >= 0; --s) {
        need_OUT[s] = need_next;
        int worst = 0;
        for (int j = 0; j < nk; ++j) {
            int cur = need_OUT[s];
            for (int n = nd - 1; n >= 0; --n) {
                const ConvLayer& c1 = rb_c1[s * nk + j][n];
                const int r1 = std::max(c1.pad, (c1.K - 1) * c1.dil - c1.pad);
                need_X[s * nk + j][n] = cur;                       // output of this dilation step (R, or OUT for the last)
                if (type1) {
                    const ConvLayer& c2 = rb_c2[s * nk + j][n];
                    const int r2 = std::max(c2.pad, (c2.K - 1) * c2.dil - c2.pad);
                    need_T1[s * nk + j][n] = cur + r2;
                    cur += r2 + r1;
                } else {
                    cur += r1;
                }
            }
            worst = std::max(worst, cur);
        }
        need_U[s] = worst;
        const ConvLayer& u = ups[s];                               // polyphase: GEMM columns are input steps
        need_q_ups[s] = (need_U[s] + u.ups - 1) / u.ups;
        need_next = need_q_ups[s] + std::max(u.pad, (u.K - 1) * u.dil - u.pad);
    }
    need_P = need_next;
}

void Hifigan::stage_dims(int T, std::vector<int>& C, std::vector<int>& L) const {
    C.resize(c.num_upsamples);
    L.resize(c.num_upsamples);
    int ch = c.upsample_initial_channel, len = T;
    for (int s = 0; s < c.num_upsamples; ++s) {
        ch /= 2;
        len = conv_transpose_out_len(ups[s], len);
        C[s] = ch;
        L[s] = len;
    }
}

size_t Hifigan::workspace_bytes(int B, int T) const {
    std::vector<int> C, L;
    stage_dims(T, C, L);
    size_t mx = 0;
    for (size_t s = 0; s < C.size(); ++s) mx = std::max(mx, (size_t)C[s] * (size_t)L[s]);
    const size_t Tp = (size_t)(T + 3) / 4 * 4;    // 16-byte aligned row pitch for the stage-0 tensors
    size_t tot = arena_bytes((size_t)B * c.upsample_initial_channel * Tp);
    tot += arena_bytes((size_t)B * c.in_channels * Tp);
    tot += 4 * arena_bytes((size_t)B * mx);
    tot += arena_bytes((size_t)B * cond.RowsPad + 64);
    return tot;
}

int Hifigan::out_len(int T) const {
    std::vector<int> C, L;
    stage_dims(T, C, L);
    return L.back();
}

int Hifigan::forward(const float* x, const float* g, int B, int T, float* wav, void* ws, size_t ws_bytes,
                     cudaStream_t st, unsigned* peak_bits, const int* lens) const {
    B200_REQUIRE(x && wav && ws, "hifigan_forward: null pointer");
    B200_REQUIRE((c.cond_channels > 0) == (g != nullptr) || c.cond_channels == 0,
                 "hifigan_forward: model has cond_channels=%d but g is null", c.cond_channels);
    B200_REQUIRE(ws_bytes >= workspace_bytes(B, T), "hifigan_forward: workspace too small");
    if (B == 0 || T == 0) return 0;
    std::vector<int> C, L;
    stage_dims(T, C, L);
    size_t mx = 0;
    for (size_t s = 0; s < C.size(); ++s) mx = std::max(mx, (size_t)C[s] * (size_t)L[s]);
    Arena ar(ws, ws_bytes);
    const int C0 = c.upsample_initial_channel;
    // The tcgen05 kernels stage activation rows with 16-byte cp.async: rows must start 16-byte aligned.  T (decoder frames)
    // is arbitrary, so the stage-0 tensors use a row pitch rounded up to 4 floats and an unaligned input is re-pitched
    // once (B x Cin x T floats, tiny) -- otherwise conv_pre / ups[0] would silently take the FP32-FMA kernel for 3 of 4 T.
    const int Tp = (T + 3) / 4 * 4;
    float* P = ar.f32((size_t)B * C0 * Tp);
    float* Xp = ar.f32((size_t)B * c.in_channels * Tp);
    float* U = ar.f32((size_t)B * mx);
    float* T1 = ar.f32((size_t)B * mx);
    float* R = ar.f32((size_t)B * mx);
    float* OUT = ar.f32((size_t)B * mx);
    float* condv = ar.f32((size_t)B * cond.RowsPad + 64);
    B200_REQUIRE(P && Xp && U && T1 && R && OUT && condv, "hifigan_forward: arena exhausted");
    const float* xin0 = x;
    int x_pitch = T;
    if (Tp != T || (reinterpret_cast<uintptr_t>(x) & 15) != 0) {
        B200_CUDA_OK(cudaMemcpy2DAsync(Xp, (size_t)Tp * sizeof(float), x, (size_t)T * sizeof(float), (size_t)T * sizeof(float),
                                       (size_t)B * c.in_channels, cudaMemcpyDeviceToDevice, st));
        xin0 = Xp;
        x_pitch = Tp;
    }
    int rc;
    const bool has_cond = c.cond_channels > 0 && g != nullptr;
    if (has_cond) {  // cond_layer(g): [B, cond, 1] -> [B, C0]
        ConvIO io;
        io.x = g; io.x_bs = c.cond_channels; io.x_cs = 1; io.Tin = 1;
        io.y = condv; io.y_bs = cond.RowsPad; io.y_cs = 1; io.Tout = 1; io.B = B;
        if ((rc = launch_conv(cond, io, st))) return rc;
    }
    {  // conv_pre (+ cond broadcast over T)
        ConvIO io;
        io.x = xin0; io.x_bs = (long long)c.in_channels * x_pitch; io.x_cs = x_pitch; io.Tin = T;
        io.y = P; io.y_bs = (long long)C0 * Tp; io.y_cs = Tp; io.Tout = T; io.B = B;
        if (has_cond) { io.cond = condv; io.cond_bs = cond.RowsPad; }
        io.lens = lens; io.rate_out = 1; io.need_out = need_P; io.rate_in = 1; io.need_in = T;   // z is defined everywhere
        if ((rc = launch_conv(conv_pre, io, st))) return rc;
    }
    const float* cur = P;
    int curC = C0, curL = T, curPitch = Tp;
    const bool type1 = c.resblock_type == 1;
    for (int s = 0; s < c.num_upsamples; ++s) {
        const int Cs = C[s], Ls = L[s];
        const long long bs = (long long)Cs * Ls;
        {  // o = ups(leaky_relu(o, 0.1))
            ConvIO io;
            io.x = cur; io.x_bs = (long long)curC * curPitch; io.x_cs = curPitch; io.Tin = curL; io.in_slope = 0.1f;
            io.y = U; io.y_bs = bs; io.y_cs = Ls; io.Tout = Ls; io.B = B;
            io.lens = lens; io.rate_in = (s == 0) ? 1 : rate[s - 1]; io.need_in = (s == 0) ? need_P : need_OUT[s - 1];
            io.rate_out = io.rate_in; io.need_out = need_q_ups[s];      // tiles run over GEMM columns = input steps
            if ((rc = launch_conv(ups[s], io, st))) return rc;
        }
        for (int j = 0; j < c.num_kernels; ++j) {
            const auto& c1 = rb_c1[s * c.num_kernels + j];
            const auto& c2 = rb_c2[s * c.num_kernels + j];
            const float* xin = U;
            int need_xin = need_U[s];
            float* pp[2] = {R, T1};  // ping-pong for ResBlock2
            for (int n = 0; n < c.num_dilations; ++n) {
                const bool last = (n == c.num_dilations - 1);
                const float* convin = xin;
                const ConvLayer* lastconv = &c1[n];
                if (type1) {  // T1 = c1(lrelu(xin))
                    ConvIO io;
                    io.x = xin; io.x_bs = bs; io.x_cs = Ls; io.Tin = Ls; io.in_slope = 0.1f;
                    io.y = T1; io.y_bs = bs; io.y_cs = Ls; io.Tout = Ls; io.B = B;
                    io.lens = lens; io.rate_in = io.rate_out = rate[s];
                    io.need_in = need_xin; io.need_out = need_T1[s * c.num_kernels + j][n];
                    if ((rc = launch_conv(c1[n], io, st))) return rc;
                    convin = T1;
                    lastconv = &c2[n];
                }
                ConvIO io;  // xnew = conv(lrelu(convin)) + xin ; MRF: OUT (+)= xnew, mean on the last resblock
                io.x = convin; io.x_bs = bs; io.x_cs = Ls; io.Tin = Ls; io.in_slope = 0.1f;
                io.res = xin; io.res_bs = bs; io.res_cs = Ls;
                io.B = B; io.Tout = Ls; io.y_bs = bs; io.y_cs = Ls;
                float* dst;
                if (last) {
                    dst = OUT;
                    if (j > 0) io.flags |= EPI_ACCUM;
                    if (j == c.num_kernels - 1) io.post_div = (float)c.num_kernels;
                } else {
                    dst = type1 ? R : pp[n & 1];
                }
                io.y = dst;
                io.lens = lens; io.rate_in = io.rate_out = rate[s];
                io.need_in = type1 ? need_T1[s * c.num_kernels + j][n] : need_xin;
                io.need_out = need_X[s * c.num_kernels + j][n];
                if ((rc = launch_conv(*lastconv, io, st))) return rc;
                xin = dst;
                need_xin = io.need_out;
            }
        }
        cur = OUT;
        curC = Cs;
        curL = Ls;
        curPitch = Ls;
        // the next stage's ups reads OUT and writes U; OUT is only rewritten by later launches
        // on the same stream, after that read has completed.
    }
    {  // tanh(conv_post(leaky_relu(o)))  -- default slope 0.01 (hifigan_generator.py:262)
        ConvIO io;
        io.x = cur; io.x_bs = (long long)curC * curPitch; io.x_cs = curPitch; io.Tin = curL; io.in_slope = 0.01f;
        io.y = wav; io.y_bs = (long long)c.out_channels * curL; io.y_cs = curL; io.Tout = curL; io.B = B;
        io.act = ACT_TANH;
        io.peak_bits = peak_bits;
        io.lens = lens; io.rate_in = io.rate_out = rate.empty() ? 1 : rate.back(); io.need_in = need_OUT.empty() ? 0 : need_OUT.back();
        io.need_out = 0;
        if (lens)   // rows may end before any tile of conv_post's fallback kernels writes them: the tail must be zero
            B200_CUDA_OK(cudaMemsetAsync(wav, 0, (size_t)B * c.out_channels * curL * sizeof(float), st));
        if ((rc = launch_conv(conv_post, io, st))) return rc;
    }
    return 0;
}

}  // namespace b200tts
