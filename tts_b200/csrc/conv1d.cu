// Generic fused conv1d as an FP32 implicit GEMM on the sm_100a FMA pipe (packed FFMA2).
//
// This one kernel carries >99% of the VITS+HiFiGAN inference FLOPs: the HiFiGAN MRF convs
// (reference: TTS/vocoder/models/hifigan_generator.py:84-99,236-265), the polyphase form of its
// ConvTranspose1d upsamplers (:207-218), the WaveNet k5 / 1x1 convs of the flow
// (TTS/tts/layers/generic/wavenet.py:94-115) and the 1x1 / k3 convs of the text encoder
// (TTS/tts/layers/glow_tts/transformer.py:109-121,290-295).
//
// Layout: activations stay in the reference's [B, C, T] layout (T contiguous).  A CTA owns a
// [CO_T rows] x [T_T time] output tile.  Input channels are streamed in chunks of 8 through a
// double-buffered shared-memory window [8][T_T + (K-1)*dil] (coalesced loads along T, prologue
// -- mask, leaky-relu -- applied once on the way in) next to the chunk's weights
// [8][K][CO_T] (cp.async).  Each lane owns TJ time steps strided by 32 (conflict-free LDS.32,
// tap shifts are plain address offsets) and CJ=16 consecutive rows (warp-uniform weight LDS.128
// broadcasts), accumulating row pairs with fma.rn.f32x2 (SASS FFMA2, x as broadcast scalar).
// Bias / conditioning / gate / residual / mask / MRF-accumulate epilogues are fused.
#include "common.cuh"
#include "engines.cuh"
#include "conv_tc.cuh"
#include "conv_tc3.cuh"

#include <stdarg.h>
#include <stdlib.h>
#include <string.h>

namespace b200tts {

// ------------------------------------------------------------------ error plumbing / counters
static thread_local char g_err[1024] = "";
unsigned long long g_launch_count = 0;

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}
const char* last_error() { return g_err; }

int upload(float** dst, const float* src, size_t n) {
    *dst = nullptr;
    if (n == 0) return 0;
    B200_CUDA_OK(cudaMalloc((void**)dst, n * sizeof(float)));
    B200_CUDA_OK(cudaMemcpy(*dst, src, n * sizeof(float), cudaMemcpyHostToDevice));
    return 0;
}

// ------------------------------------------------------------------ device helpers
constexpr int CI_MAX = 16;  // CinPad granularity (largest input-channel chunk of any instantiation)

typedef unsigned long long u64;

__device__ __forceinline__ void ffma2(u64& d, u64 a, float x) {
    u64 xx;
    asm("mov.b64 %0, {%1, %1};" : "=l"(xx) : "f"(x));
    asm("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(d) : "l"(a), "l"(xx));
}
__device__ __forceinline__ void unpack2(u64 v, float& lo, float& hi) {
    asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ u64 pack2(float lo, float hi) {
    u64 v;
    asm("mov.b64 %0, {%1, %2};" : "=l"(v) : "f"(lo), "f"(hi));
    return v;
}
__device__ __forceinline__ void cp_async16(float* smem_dst, const float* gsrc) {
    unsigned s = (unsigned)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(s), "l"(gsrc));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }

struct ConvKArgs {
    const float* x; long long x_bs; int x_cs; int Tin;
    const float* xmask; long long xmask_bs; float in_slope;
    const float* w; const float* bias; const float* cond; long long cond_bs;
    int Cin, CinPad, K, dil, pad, Rows, ups, Tq;
    float* y; long long y_bs; int y_cs; int Tout;
    const float* res; long long res_bs; int res_cs;
    const float* ymask; long long ymask_bs;
    float* y2; long long y2_bs; int y2_cs; int split;
    float scale; float post_div; int act; float act_param; int flags;
    int XS;
    const int* lens; int rate_out, need_out, rate_in, need_in;
};

enum : int { KEPI_GENERIC = 0, KEPI_GATE = 1, KEPI_TANH = 2, KEPI_PLAIN = 3 };

// CJ rows x TJ time steps per lane, WCO x WT warps, CIC input channels per stage, EPI epilogue family.
// KG > 1: intra-CTA split-K for launch-starved shapes (text encoder / duration predictor: 64 frames x 32 utterances
// give only 96 CTAs of 4 warps) -- KG warp groups each own a double-buffered stage and every KG-th channel chunk of
// the SAME output tile; their accumulators are summed through shared memory in a fixed order (deterministic).
template <int CJ, int TJ, int WCO, int WT, int CIC, int EPI, int KG = 1>
__global__ void __launch_bounds__(32 * WCO * WT * KG, (KG > 1) ? 1 : ((WCO * WT >= 8) ? 2 : 3)) conv1d_kernel(const ConvKArgs a) {
    constexpr int CO_T = CJ * WCO, T_T = 32 * TJ * WT, NT = 32 * WCO * WT;
    extern __shared__ __align__(16) float smem[];
    const int XS = a.XS;
    const int wchunk = CIC * a.K * CO_T;
    const int kg = (KG > 1) ? (int)(threadIdx.x / NT) : 0;              // split-K group of this warp
    const int stage_floats = 2 * CIC * XS + 2 * wchunk;
    float* xs0 = smem + (size_t)kg * stage_floats;
    float* ws0 = xs0 + 2 * CIC * XS;
    const int tid = threadIdx.x % NT, lane = tid & 31, warp = tid >> 5;   // group-local thread / warp index
    const int wco = warp % WCO, wt = warp / WCO;
    auto group_sync = [&]() {
        if constexpr (KG > 1) asm volatile("bar.sync %0, %1;" ::"r"(kg + 1), "r"(NT) : "memory");
        else __syncthreads();
    };
    const int b = blockIdx.z, tile_co = blockIdx.y;
    const int q0 = blockIdx.x * T_T;
    const int tin0 = q0 - a.pad;
    const float* xb = a.x + b * a.x_bs;
    const float* mb = a.xmask ? a.xmask + b * a.xmask_bs : nullptr;
    const float* wg = a.w + (size_t)tile_co * a.CinPad * a.K * CO_T;
    const int nchunks = (a.Cin + CIC - 1) / CIC;   // CinPad is a multiple of CI_MAX >= CIC; skip all-zero chunks
    const float slope = a.in_slope;

    auto load_chunk = [&](int chunk, int buf) {
        const float* src = wg + (size_t)chunk * wchunk;
        float* dst = ws0 + buf * wchunk;
        for (int i = tid * 4; i < wchunk; i += NT * 4) cp_async16(dst + i, src + i);
        cp_async_commit();
        float* xd = xs0 + buf * CIC * XS;
        const int c0 = chunk * CIC;
        for (int i = tid; i < XS; i += NT) {
            const int t = tin0 + i;
            const bool tok = (t >= 0) && (t < a.Tin);
            float m = 1.f;
            if (tok && mb) m = __ldg(mb + t);
#pragma unroll
            for (int h = 0; h < CIC; h += 8) {
                float v[8];
#pragma unroll
                for (int ci = 0; ci < 8; ++ci) {
                    v[ci] = 0.f;
                    if (tok && (c0 + h + ci) < a.Cin) v[ci] = __ldg(xb + (long long)(c0 + h + ci) * a.x_cs + t);
                }
#pragma unroll
                for (int ci = 0; ci < 8; ++ci) {
                    float u = v[ci] * m;
                    u = u > 0.f ? u : u * slope;
                    xd[(h + ci) * XS + i] = u;
                }
            }
        }
    };

    u64 acc[CJ / 2][TJ];
#pragma unroll
    for (int p = 0; p < CJ / 2; ++p)
#pragma unroll
        for (int j = 0; j < TJ; ++j) acc[p][j] = 0ull;

    if (kg < nchunks) load_chunk(kg, 0);
    cp_async_wait_all();
    group_sync();

    const int K = a.K, dil = a.dil;
    for (int ch = kg, it = 0; ch < nchunks; ch += KG, ++it) {
        const int buf = it & 1;
        if (ch + KG < nchunks) load_chunk(ch + KG, buf ^ 1);
        const float* xr = xs0 + buf * CIC * XS + wt * 32 * TJ + lane;
        const float* wr = ws0 + buf * wchunk + wco * CJ;
#pragma unroll 1
        for (int ci = 0; ci < CIC; ++ci) {
            const float* xp = xr + ci * XS;
            const ulonglong2* wp = reinterpret_cast<const ulonglong2*>(wr + ci * K * CO_T);
#pragma unroll 1
            for (int k = 0; k < K; ++k) {
                float xv[TJ];
#pragma unroll
                for (int j = 0; j < TJ; ++j) xv[j] = xp[32 * j];
                u64 wv[CJ / 2];
#pragma unroll
                for (int p = 0; p < CJ / 4; ++p) {
                    const ulonglong2 t2 = wp[p];
                    wv[2 * p] = t2.x;
                    wv[2 * p + 1] = t2.y;
                }
#pragma unroll
                for (int j = 0; j < TJ; ++j)
#pragma unroll
                    for (int p = 0; p < CJ / 2; ++p) ffma2(acc[p][j], wv[p], xv[j]);
                xp += dil;
                wp += CO_T / 4;
            }
        }
        cp_async_wait_all();
        group_sync();
    }

    if constexpr (KG > 1) {
        // fixed-order sum of the groups' partial accumulators (group 0 += group 1 += ...), through the stage memory
        __syncthreads();
        u64* red = reinterpret_cast<u64*>(smem);
        if (kg > 0) {
#pragma unroll
            for (int p = 0; p < CJ / 2; ++p)
#pragma unroll
                for (int j = 0; j < TJ; ++j) red[(((size_t)(kg - 1) * (CJ / 2) + p) * TJ + j) * NT + tid] = acc[p][j];
        }
        __syncthreads();
        if (kg > 0) return;
#pragma unroll
        for (int g2 = 1; g2 < KG; ++g2)
#pragma unroll
            for (int p = 0; p < CJ / 2; ++p)
#pragma unroll
                for (int j = 0; j < TJ; ++j) {
                    float v0, v1, w0, w1;
                    unpack2(acc[p][j], v0, v1);
                    unpack2(red[(((size_t)(g2 - 1) * (CJ / 2) + p) * TJ + j) * NT + tid], w0, w1);
                    acc[p][j] = pack2(v0 + w0, v1 + w1);
                }
    }

    // ---------------------------------------------------------------- epilogue
    const int row_base = tile_co * CO_T + wco * CJ;
    const int qb = q0 + wt * 32 * TJ + lane;
    if (EPI == KEPI_GATE) {
        // rows (2p, 2p+1) = (tanh half, sigmoid half) of output row row_base/2 + p   (wavenet.py:6-13)
#pragma unroll
        for (int p = 0; p < CJ / 2; ++p) {
            const int r0 = row_base + 2 * p;
            if (r0 + 1 < a.Rows) {
                float b0 = a.bias[r0], b1 = a.bias[r0 + 1];
                if (a.cond) { b0 += __ldg(a.cond + b * a.cond_bs + r0); b1 += __ldg(a.cond + b * a.cond_bs + r0 + 1); }
                float* yrow = a.y + b * a.y_bs + (long long)(r0 >> 1) * a.y_cs;
#pragma unroll
                for (int j = 0; j < TJ; ++j) {
                    const int q = qb + 32 * j;
                    float v0, v1;
                    unpack2(acc[p][j], v0, v1);
                    v0 += b0; v1 += b1;
                    if (q < a.Tout) yrow[q] = tanhf(v0) * (1.f / (1.f + expf(-v1)));
                }
            }
        }
        return;
    }
    if (EPI == KEPI_TANH) {   // conv_post: y = tanh(acc + bias)   (hifigan_generator.py:263-264)
#pragma unroll
        for (int p = 0; p < CJ / 2; ++p) {
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                const int r = row_base + 2 * p + h;
                if (r < a.Rows) {
                    const float bb = a.bias[r];
                    float* yrow = a.y + b * a.y_bs + (long long)r * a.y_cs;
#pragma unroll
                    for (int j = 0; j < TJ; ++j) {
                        const int q = qb + 32 * j;
                        float v0, v1;
                        unpack2(acc[p][j], v0, v1);
                        if (q < a.Tout) yrow[q] = tanhf((h ? v1 : v0) + bb);
                    }
                }
            }
        }
        return;
    }
    if (EPI == KEPI_PLAIN) {   // y = act(acc + bias + cond) [* mask]   -- no residual / accumulate / upsampling
        const bool relu_p = a.act == ACT_RELU;
        const bool logc_p = a.act == ACT_LOGCLAMP;
        float mkp[TJ];
#pragma unroll
        for (int j = 0; j < TJ; ++j) {
            const int q = qb + 32 * j;
            mkp[j] = (a.ymask && q < a.Tout) ? __ldg(a.ymask + b * a.ymask_bs + q) : 1.f;
        }
#pragma unroll
        for (int p = 0; p < CJ / 2; ++p) {
            const int r0 = row_base + 2 * p;
            float b0 = 0.f, b1 = 0.f;
            if (r0 < a.Rows) { b0 = a.bias[r0]; if (a.cond) b0 += __ldg(a.cond + b * a.cond_bs + r0); }
            if (r0 + 1 < a.Rows) { b1 = a.bias[r0 + 1]; if (a.cond) b1 += __ldg(a.cond + b * a.cond_bs + r0 + 1); }
            float* y0 = a.y + b * a.y_bs + (long long)r0 * a.y_cs;
            float* y1 = y0 + a.y_cs;
#pragma unroll
            for (int j = 0; j < TJ; ++j) {
                const int q = qb + 32 * j;
                float v0, v1;
                unpack2(acc[p][j], v0, v1);
                v0 += b0; v1 += b1;
                if (relu_p) { v0 = fmaxf(v0, 0.f); v1 = fmaxf(v1, 0.f); }
                if (logc_p) { v0 = logf(fmaxf(v0, a.act_param)); v1 = logf(fmaxf(v1, a.act_param)); }
                v0 *= mkp[j]; v1 *= mkp[j];
                if (q < a.Tout) {
                    if (r0 < a.Rows) y0[q] = v0;
                    if (r0 + 1 < a.Rows) y1[q] = v1;
                }
            }
        }
        return;
    }
    // generic: v = act(acc + bias + cond) [*m] [+res] *scale [+y_old] [/div] [*m]; all loads are issued before
    // any store (res / y_old may alias y only element-for-element, never across threads)
    const int ups = a.ups;
    const bool relu = a.act == ACT_RELU;
    const bool split = (a.flags & EPI_SPLIT) != 0;
    float mk[TJ];
    int tq[TJ];
#pragma unroll
    for (int j = 0; j < TJ; ++j) {
        tq[j] = (qb + 32 * j) * ups;
        mk[j] = 1.f;
        if (a.ymask && ups == 1 && tq[j] < a.Tout) mk[j] = __ldg(a.ymask + b * a.ymask_bs + tq[j]);
    }
    // per-row destination: recomputed per phase instead of kept in registers (16 rows x 2 pointers would spill)
    auto rowinfo = [&](int i, float*& yp, const float*& rp, bool& accum, bool& mpost, int& tlim) -> bool {
        const int r = row_base + i;
        int chn = r, ph = 0;
        if (ups > 1) { chn = r / ups; ph = r - chn * ups; }
        accum = (a.flags & EPI_ACCUM) != 0;
        mpost = (a.flags & EPI_MASK_POST) != 0;
        yp = a.y + b * a.y_bs + (long long)chn * a.y_cs + ph;
        if (split) {
            if (chn < a.split) { accum = true; mpost = true; }
            else { yp = a.y2 + b * a.y2_bs + (long long)(chn - a.split) * a.y2_cs; accum = (a.flags & EPI_ACCUM2) != 0; mpost = false; }
        }
        rp = a.res ? a.res + b * a.res_bs + (long long)chn * a.res_cs + ph : nullptr;
        tlim = a.Tout - ph;   // element (q*ups + ph) exists iff q*ups < Tout - ph
        return r < a.Rows;
    };
    const bool mpre = (a.flags & EPI_MASK_PRE) != 0;
    // phase 1: bias / cond / activation / pre-mask (registers only)
#pragma unroll
    for (int p = 0; p < CJ / 2; ++p) {
        const int r0 = row_base + 2 * p;
        float b0 = 0.f, b1 = 0.f;
        if (r0 < a.Rows) { b0 = a.bias[r0]; if (a.cond) b0 += __ldg(a.cond + b * a.cond_bs + r0); }
        if (r0 + 1 < a.Rows) { b1 = a.bias[r0 + 1]; if (a.cond) b1 += __ldg(a.cond + b * a.cond_bs + r0 + 1); }
#pragma unroll
        for (int j = 0; j < TJ; ++j) {
            float v0, v1;
            unpack2(acc[p][j], v0, v1);
            v0 += b0; v1 += b1;
            if (relu) { v0 = fmaxf(v0, 0.f); v1 = fmaxf(v1, 0.f); }
            if (mpre) { v0 *= mk[j]; v1 *= mk[j]; }
            acc[p][j] = pack2(v0, v1);
        }
    }
    // phase 2: residual (all loads first)
    if (a.res) {
#pragma unroll
        for (int p = 0; p < CJ / 2; ++p) {
            float *yp0, *yp1; const float *rp0, *rp1; bool ac0, ac1, mp0, mp1; int tl0, tl1;
            const bool ok0 = rowinfo(2 * p, yp0, rp0, ac0, mp0, tl0), ok1 = rowinfo(2 * p + 1, yp1, rp1, ac1, mp1, tl1);
#pragma unroll
            for (int j = 0; j < TJ; ++j) {
                float v0, v1, r0v = 0.f, r1v = 0.f;
                if (ok0 && tq[j] < tl0) r0v = rp0[tq[j]];
                if (ok1 && tq[j] < tl1) r1v = rp1[tq[j]];
                unpack2(acc[p][j], v0, v1);
                acc[p][j] = pack2(v0 + r0v, v1 + r1v);
            }
        }
    }
    // phase 3: scale, accumulate into the destination (all loads first)
    const float scale = a.scale;
    if (split || (a.flags & EPI_ACCUM)) {
#pragma unroll
        for (int p = 0; p < CJ / 2; ++p) {
            float *yp0, *yp1; const float *rp0, *rp1; bool ac0, ac1, mp0, mp1; int tl0, tl1;
            const bool ok0 = rowinfo(2 * p, yp0, rp0, ac0, mp0, tl0), ok1 = rowinfo(2 * p + 1, yp1, rp1, ac1, mp1, tl1);
#pragma unroll
            for (int j = 0; j < TJ; ++j) {
                float v0, v1, o0 = 0.f, o1 = 0.f;
                if (ac0 && ok0 && tq[j] < tl0) o0 = yp0[tq[j]];
                if (ac1 && ok1 && tq[j] < tl1) o1 = yp1[tq[j]];
                unpack2(acc[p][j], v0, v1);
                acc[p][j] = pack2(v0 * scale + o0, v1 * scale + o1);
            }
        }
    } else if (scale != 1.f) {
#pragma unroll
        for (int p = 0; p < CJ / 2; ++p)
#pragma unroll
            for (int j = 0; j < TJ; ++j) {
                float v0, v1;
                unpack2(acc[p][j], v0, v1);
                acc[p][j] = pack2(v0 * scale, v1 * scale);
            }
    }
    // phase 4: mean / post-mask / store
    const float div = a.post_div;
#pragma unroll
    for (int p = 0; p < CJ / 2; ++p) {
        float *yp0, *yp1; const float *rp0, *rp1; bool ac0, ac1, mp0, mp1; int tl0, tl1;
        const bool ok0 = rowinfo(2 * p, yp0, rp0, ac0, mp0, tl0), ok1 = rowinfo(2 * p + 1, yp1, rp1, ac1, mp1, tl1);
#pragma unroll
        for (int j = 0; j < TJ; ++j) {
            float v0, v1;
            unpack2(acc[p][j], v0, v1);
            if (div != 1.f) { v0 = v0 / div; v1 = v1 / div; }
            if (mp0) v0 *= mk[j];
            if (mp1) v1 *= mk[j];
            if (ok0 && tq[j] < tl0) yp0[tq[j]] = v0;
            if (ok1 && tq[j] < tl1) yp1[tq[j]] = v1;
        }
    }
}

// ------------------------------------------------------------------ host: packing
static inline int round_up(int v, int m) { return (v + m - 1) / m * m; }

void free_conv(ConvLayer& L) {
    if (L.w) cudaFree(L.w);
    if (L.bias) cudaFree(L.bias);
    if (L.w_tc) cudaFree(L.w_tc);
    if (L.w_tcg) cudaFree(L.w_tcg);
    L.w = L.bias = L.w_tc = L.w_tcg = nullptr;
}

// Host twin of the single-pass producers' cvt.rna.tf32.f32: round a finite value to the nearest TF32 value, ties away
// from zero (sign-magnitude, so adding half an ulp to the bits and truncating does it); inf / NaN pass through.
static float tf32_rna(float v) {
    uint32_t u;
    memcpy(&u, &v, 4);
    if ((u & 0x7F800000u) != 0x7F800000u) { u += 0x1000u; u &= 0xFFFFE000u; }
    memcpy(&v, &u, 4);
    return v;
}
// One weight of a tcgen05 tap block: 3 passes -> hi (TF32 truncation) at hi[i], the exact remainder at lo[i];
// 1 pass -> the TF32-rounded value at hi[i] (there is no lo half)
static inline void put_tc_weight(float v, int passes, float* hi, float* lo, size_t i) {
    if (passes == 1) { hi[i] = tf32_rna(v); return; }
    uint32_t u;
    memcpy(&u, &v, 4);
    u &= 0xFFFFE000u;
    float h;
    memcpy(&h, &u, 4);
    hi[i] = h;
    lo[i] = v - h;
}

// Wl(r, ci, k): logical weights already expressed as a correlation-form conv with `rows` GEMM rows
static int pack_rows(ConvLayer& L, const std::vector<float>& Wl, const std::vector<float>& bl, int rows, int Cin,
                     int K, int tc_passes) {
    B200_REQUIRE(tc_passes == 1 || tc_passes == 3, "conv pack: tc_passes must be 1 or 3, got %d", tc_passes);
    L.tc_passes = tc_passes;
    const int halves = tc_passes == 1 ? 1 : 2;     // {hi, lo} or {w} per tap block
    L.Rows = rows;
    L.co_tile = rows >= 64 ? 64 : 32;
    L.RowsPad = round_up(rows, L.co_tile);
    L.Cin = Cin;
    L.CinPad = round_up(Cin, CI_MAX);
    L.K = K;
    const int T = L.co_tile, ntile = L.RowsPad / T;
    std::vector<float> P((size_t)ntile * L.CinPad * K * T, 0.f);
    for (int r = 0; r < rows; ++r) {
        const int tile = r / T, col = r % T;
        for (int ci = 0; ci < Cin; ++ci)
            for (int k = 0; k < K; ++k)
                P[(((size_t)tile * L.CinPad + ci) * K + k) * T + col] = Wl[((size_t)r * Cin + ci) * K + k];
    }
    std::vector<float> bp(L.RowsPad, 0.f);
    for (int r = 0; r < rows; ++r) bp[r] = bl[r];
    if (upload(&L.w, P.data(), P.size())) return 2;
    if (upload(&L.bias, bp.data(), bp.size())) return 2;
    // tcgen05 packing (3xTF32 hi/lo split, or single-pass TF32) for layers the tensor-core kernel can take
    // rows >= 32: tiles of 128 zero-padded rows (tcgen05 M = 128); exactly 32 / 64 rows additionally get the grouped
    // packing below (no padding), which the dispatcher prefers; fewer rows run on the FP32-FMA kernel
    L.tc_n = 0;
    if (rows >= 32) L.tc_n = 128;
    if (L.tc_n && rows >= 16 && Cin >= 8) {
        using namespace tc;
        const int N = L.tc_n, nt = (rows + N - 1) / N, nchunk = (Cin + KC - 1) / KC;
        const size_t blk = (size_t)halves * NSLAB * N * 4;
        std::vector<float> Q((size_t)nt * nchunk * K * blk, 0.f);
        for (int tile = 0; tile < nt; ++tile)
            for (int c = 0; c < nchunk; ++c)
                for (int k = 0; k < K; ++k) {
                    float* dst = Q.data() + (((size_t)tile * nchunk + c) * K + k) * blk;
                    for (int s2 = 0; s2 < NSLAB; ++s2)
                        for (int n = 0; n < N; ++n)
                            for (int i = 0; i < 4; ++i) {
                                const int r = tile * N + n, ci = c * KC + 4 * s2 + i;
                                const float v = (ci < Cin && r < rows) ? Wl[((size_t)r * Cin + ci) * K + k] : 0.f;
                                put_tc_weight(v, tc_passes, dst, dst + (size_t)NSLAB * N * 4, ((size_t)s2 * N + n) * 4 + i);
                            }
                }
        if (upload(&L.w_tc, Q.data(), Q.size())) return 2;
    } else {
        L.tc_n = 0;
    }
    // grouped packing for exactly 32 / 64 rows (conv_tc3.cuh, grouped mode): MMA row m = g * rows + co holds channel co
    // and tap group g (a TMEM lane quarter = one group); tap block j carries tap G*j + g (zero beyond K)
    L.tc_grp = 0;
    if (L.ups == 1 && (rows == 32 || rows == 64) && Cin >= 8) {
        using namespace tc;
        const int G = 128 / rows, J = (K + G - 1) / G, nchunk = (Cin + KC - 1) / KC;
        const size_t blk = (size_t)halves * NSLAB * 128 * 4;
        std::vector<float> Q((size_t)nchunk * J * blk, 0.f);
        for (int c = 0; c < nchunk; ++c)
            for (int j = 0; j < J; ++j) {
                float* dst = Q.data() + ((size_t)c * J + j) * blk;
                for (int s2 = 0; s2 < NSLAB; ++s2)
                    for (int m = 0; m < 128; ++m)
                        for (int i = 0; i < 4; ++i) {
                            const int g = m / rows, co = m % rows;
                            const int k = G * j + g, ci = c * KC + 4 * s2 + i;
                            const float v = (ci < Cin && k < K) ? Wl[((size_t)co * Cin + ci) * K + k] : 0.f;
                            put_tc_weight(v, tc_passes, dst, dst + (size_t)NSLAB * 128 * 4, ((size_t)s2 * 128 + m) * 4 + i);
                        }
            }
        if (upload(&L.w_tcg, Q.data(), Q.size())) return 2;
        L.tc_grp = G;
    }
    return 0;
}

int pack_conv(ConvLayer& L, const float* w, const float* bias, int Cout, int Cin, int K, int dil, int pad,
              int gate_half, const int* in_perm, const int* out_perm, int tc_passes) {
    B200_REQUIRE(w != nullptr && Cout > 0 && Cin > 0 && K > 0, "pack_conv: bad arguments");
    B200_REQUIRE(gate_half == 0 || 2 * gate_half == Cout, "pack_conv: gate_half must be Cout/2");
    std::vector<float> Wl((size_t)Cout * Cin * K), bl(Cout, 0.f);
    for (int r = 0; r < Cout; ++r) {
        int rn = r;
        if (gate_half > 0) rn = (r < gate_half) ? 2 * r : 2 * (r - gate_half) + 1;
        if (out_perm) rn = out_perm[r];
        for (int ci = 0; ci < Cin; ++ci) {
            const int cn = in_perm ? in_perm[ci] : ci;
            for (int k = 0; k < K; ++k) Wl[((size_t)rn * Cin + cn) * K + k] = w[((size_t)r * Cin + ci) * K + k];
        }
        if (bias) bl[rn] = bias[r];
    }
    L.dil = dil;
    L.pad = pad;
    L.ups = 1;
    return pack_rows(L, Wl, bl, Cout, Cin, K, tc_passes);
}

int pack_conv_transpose(ConvLayer& L, const float* w, const float* bias, int Cin, int Cout, int Kt, int s, int p,
                        int tc_passes) {
    // y[co, q*s+ph] = sum_ci sum_m x[ci, q-m] * w[ci, co, ph + p + m*s]   (0 <= ph+p+m*s < Kt)
    B200_REQUIRE(w != nullptr && s >= 1 && Kt >= 1, "pack_conv_transpose: bad arguments");
    auto floordiv = [](int a, int b) { return (a >= 0) ? a / b : -((-a + b - 1) / b); };
    const int m_lo = -floordiv(s - 1 + p, s);  // ceil(-(s-1+p)/s)
    const int m_hi = floordiv(Kt - 1 - p, s);
    const int K = m_hi - m_lo + 1;
    B200_REQUIRE(K >= 1, "pack_conv_transpose: empty tap range");
    const int rows = Cout * s;
    std::vector<float> Wl((size_t)rows * Cin * K, 0.f), bl(rows, 0.f);
    for (int co = 0; co < Cout; ++co)
        for (int ph = 0; ph < s; ++ph) {
            const int r = co * s + ph;
            if (bias) bl[r] = bias[co];
            for (int kk = 0; kk < K; ++kk) {
                const int m = m_hi - kk;
                const int kt = ph + p + m * s;
                if (kt < 0 || kt >= Kt) continue;
                for (int ci = 0; ci < Cin; ++ci)
                    Wl[((size_t)r * Cin + ci) * K + kk] = w[((size_t)ci * Cout + co) * Kt + kt];
            }
        }
    L.dil = 1;
    L.pad = m_hi;
    L.ups = s;
    L.tr_kernel = Kt;
    L.tr_pad = p;
    return pack_rows(L, Wl, bl, rows, Cin, K, tc_passes);
}

// ------------------------------------------------------------------ single-output-row conv (HiFiGAN conv_post)
// y[b, 0, t] = act(bias + sum_ci sum_k w[ci, k] * lrelu(x[b, ci, t + k - pad])), K taps, dilation 1.  One output row has
// no reuse across rows, so this is a pure streaming kernel: each thread owns four consecutive samples and reads its
// window as aligned float4 (neighbouring threads' overlaps are L1 hits), 4*K FMAs per channel.  HBM-bound by the x read
// (Cin * 4 B per output sample).  Reference: hifigan_generator.py:262-264.
template <int K>
__global__ void __launch_bounds__(256) conv1d_row1_kernel(const float* __restrict__ x, long long x_bs, int x_cs, int Cin,
                                                          int T, const float* __restrict__ w, int w_stride,
                                                          const float* __restrict__ bias, float slope, int act,
                                                          float* __restrict__ y, long long y_bs,
                                                          unsigned* __restrict__ peak_bits, const int* __restrict__ lens,
                                                          int rate, int need_out, int need_in) {
    constexpr int PAD = (K - 1) / 2, NL = (4 + 4 + (K - 1 - PAD) + 3) / 4;   // float4 loads covering [t0 - 4, t0 + 4 + K-1-PAD)
    extern __shared__ float ws[];
    for (int i = threadIdx.x; i < Cin * K; i += blockDim.x) ws[i] = w[(size_t)i * w_stride];
    __syncthreads();
    const int b = blockIdx.y;
    // ragged batch: row b is computed below Tb only (a multiple of 4) and samples from Tb on are written as zeros, so the
    // padded tail of the waveform is clean; the input holds data below Ti (its producer's extent) and reads as zero beyond
    int Tb = T, Ti = T;
    if (lens) {
        const long long base = (long long)lens[b] * rate;
        const long long e = (base + need_out + 3) / 4 * 4, ei = (base + need_in + 3) / 4 * 4;
        Tb = (int)(e < (long long)T ? (e > 0 ? e : 0) : (long long)T);
        Ti = (int)(ei < (long long)T ? (ei > 0 ? ei : 0) : (long long)T);
    }
    if ((int)(blockIdx.x * blockDim.x) * 4 >= Tb && !peak_bits) {        // whole block beyond the row: zero fill and leave
        const int tz = (blockIdx.x * blockDim.x + threadIdx.x) * 4;
        if (tz < T) *reinterpret_cast<float4*>(y + b * y_bs + tz) = make_float4(0.f, 0.f, 0.f, 0.f);
        return;
    }
    const int t0 = (blockIdx.x * blockDim.x + threadIdx.x) * 4;
    const bool valid = t0 < Tb;
    if (!valid && t0 < T) *reinterpret_cast<float4*>(y + b * y_bs + t0) = make_float4(0.f, 0.f, 0.f, 0.f);
    if (!valid && !peak_bits) return;
    float4 o = make_float4(0.f, 0.f, 0.f, 0.f);
    if (valid) {
        const float* xb = x + b * x_bs + t0;
        float acc[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll 4
        for (int ci = 0; ci < Cin; ++ci) {
            const float* xr = xb + (long long)ci * x_cs;
            float win[4 * NL];
#pragma unroll
            for (int l = 0; l < NL; ++l) {
                const int t = t0 - 4 + 4 * l;
                float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
                if (t >= 0 && t < Ti) v = __ldg(reinterpret_cast<const float4*>(xr - 4 + 4 * l));   // Ti % 4 == 0: all in or all out
                win[4 * l] = v.x; win[4 * l + 1] = v.y; win[4 * l + 2] = v.z; win[4 * l + 3] = v.w;
            }
#pragma unroll
            for (int i = 0; i < 4 * NL; ++i) win[i] = win[i] > 0.f ? win[i] : win[i] * slope;
#pragma unroll
            for (int k = 0; k < K; ++k) {
                const float wk = ws[ci * K + k];
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[j] = fmaf(wk, win[4 - PAD + j + k], acc[j]);
            }
        }
        const float bv = bias[0];
        float* po = &o.x;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            float u = acc[j] + bv;
            if (act == ACT_TANH) u = tanhf(u);
            po[j] = u;
        }
        *reinterpret_cast<float4*>(y + b * y_bs + t0) = o;
    }
    if (peak_bits) {   // save_wav's max|wav| (numpy_transforms.py:439) folded into the store: one atomic per warp
        float m = fmaxf(fmaxf(fabsf(o.x), fabsf(o.y)), fmaxf(fabsf(o.z), fabsf(o.w)));
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, off));
        if ((threadIdx.x & 31) == 0 && m > 0.f) atomicMax(peak_bits, __float_as_uint(m));
    }
}

// ------------------------------------------------------------------ host: launch
template <int CJ, int TJ, int WCO, int WT, int CIC, int EPI, int KG = 1>
static int launch_variant(const ConvKArgs& ka, int B, int RowsPad, cudaStream_t st) {
    constexpr int CO_T = CJ * WCO, T_T = 32 * TJ * WT, NT = 32 * WCO * WT * KG;
    ConvKArgs a = ka;
    a.XS = round_up(T_T + (a.K - 1) * a.dil, 4);
    size_t smem = (size_t)KG * (2 * CIC * a.XS + 2 * CIC * a.K * CO_T) * sizeof(float);
    if (KG > 1) smem = std::max(smem, (size_t)(KG - 1) * (CJ / 2) * TJ * (NT / KG) * sizeof(u64));
    B200_REQUIRE(smem <= 227 * 1024, "conv1d: K=%d dil=%d needs %zu B of shared memory", a.K, a.dil, smem);
    static DeviceOnce attr_once;   // one per template instantiation
    if (int rc = device_once(attr_once, nullptr, [](int) -> int {
            B200_CUDA_OK(cudaFuncSetAttribute(conv1d_kernel<CJ, TJ, WCO, WT, CIC, EPI, KG>,
                                              cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
            return 0;
        })) return rc;
    dim3 grid((a.Tq + T_T - 1) / T_T, RowsPad / CO_T, B);
    B200_REQUIRE(grid.y <= 65535 && grid.z <= 65535, "conv1d: grid too large");
    conv1d_kernel<CJ, TJ, WCO, WT, CIC, EPI, KG><<<grid, NT, smem, st>>>(a);
    count_launch();
    dispatch_note(DISPATCH_FMA);
    B200_CUDA_OK(cudaGetLastError());
    return 0;
}

template <int CIC, int EPI>
static int launch_tiles(const ConvKArgs& a, int co_tile, int B, int RowsPad, cudaStream_t st) {
    const bool small_t = a.Tq <= 128;
    if (co_tile == 64) {
        if constexpr (EPI == KEPI_PLAIN) {
            // launch-starved shape (fewer CTAs than SMs, long channel loop): split the channel chunks over 4 warp groups
            static int splitk = -1;
            if (splitk < 0) { const char* e = getenv("B200TTS_NO_SPLITK"); splitk = (e && atoi(e)) ? 0 : 1; }
            const long long ctas = (long long)((a.Tq + 63) / 64) * (RowsPad / 64) * B;
            const int nchunks = (a.Cin + CIC - 1) / CIC;
            const size_t smem4 = (size_t)4 * (2 * CIC * round_up(64 + (a.K - 1) * a.dil, 4) + 2 * CIC * a.K * 64) * sizeof(float);
            if (splitk && small_t && ctas <= 160 && nchunks >= 8 && smem4 <= 200 * 1024)
                return launch_variant<16, 2, 4, 1, CIC, EPI, 4>(a, B, RowsPad, st);
        }
        if (small_t) return launch_variant<16, 2, 4, 1, CIC, EPI>(a, B, RowsPad, st);
        return launch_variant<16, 4, 4, 2, CIC, EPI>(a, B, RowsPad, st);
    }
    if (small_t) return launch_variant<16, 2, 2, 2, CIC, EPI>(a, B, RowsPad, st);
    return launch_variant<16, 4, 2, 4, CIC, EPI>(a, B, RowsPad, st);
}

template <int EPI>
static int launch_cic(const ConvKArgs& a, int co_tile, int B, int RowsPad, cudaStream_t st) {
    // keep the work per pipeline stage roughly constant: CIC * K ~ 48..112 tap-steps
    if (a.K >= 9) return launch_tiles<8, EPI>(a, co_tile, B, RowsPad, st);
    return launch_tiles<16, EPI>(a, co_tile, B, RowsPad, st);
}

// ------------------------------------------------------------------ dispatch log (debug / tests)
static thread_local std::vector<int>* t_dispatch = nullptr;
void dispatch_begin() { delete t_dispatch; t_dispatch = new std::vector<int>(); }
int dispatch_end(int* ids, int cap) {
    if (!t_dispatch) return 0;
    const int n = (int)t_dispatch->size();
    for (int i = 0; i < n && i < cap; ++i) ids[i] = (*t_dispatch)[i];
    delete t_dispatch;
    t_dispatch = nullptr;
    return n;
}
void dispatch_note(int id) { if (t_dispatch) t_dispatch->push_back(id); }

// tcgen05 path: returns -1 when the layer / shape / epilogue is not eligible (caller falls through to the FMA kernel)
// Per-device state of the tcgen05 path: the pipeline-timeout flag lives in mapped pinned host memory (the kernels
// write it with a system-scope store), so every later launch on that device reads it WITHOUT a synchronisation and
// fails loudly instead of returning garbage audio.
struct TcDevice { int* err = nullptr; int num_sms = 0; };
static TcDevice g_tc_dev[MAX_DEVICES];
static DeviceOnce g_tc_once;

// launch with programmatic stream serialization: the kernel may be scheduled while its predecessor drains (the kernel
// itself waits with griddepcontrol.wait before touching activations).  B200TTS_NO_PDL=1 restores plain launches.
static cudaError_t launch_tc3(tc3::Tc3Kernel k, int grid, size_t smem, cudaStream_t st, const tc3::Tc3Args& t) {
    static int pdl = -1;
    if (pdl < 0) { const char* e = getenv("B200TTS_NO_PDL"); pdl = (e && atoi(e)) ? 0 : 1; }
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)grid);
    cfg.blockDim = dim3(tc3::NTHREADS2);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at;
    cfg.numAttrs = pdl ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, k, t);
}
// ragged batches: the prefix table lives behind everything else in dynamic shared memory (when it still fits)
static void set_ragged(tc3::Tc3Args& t, const ConvKArgs& a, size_t& smem) {
    t.lens = nullptr; t.rate_q = 1; t.need_q = 0; t.rate_in = 1; t.need_in = 0; t.pref_off = 0;
    if (!a.lens) return;
    const size_t off = (smem + 15) / 16 * 16, extra = tc3::ragged_table_bytes(t.B);
    if (off + extra > 227 * 1024) return;           // enormous batch: fall back to the dense schedule (still correct)
    t.lens = a.lens; t.rate_q = a.rate_out; t.need_q = a.need_out; t.rate_in = a.rate_in; t.need_in = a.need_in;
    t.pref_off = (int)off;
    smem = off + extra;
}

static int try_launch_tc(const ConvLayer& L, const ConvIO& io, const ConvKArgs& a, cudaStream_t st) {
    static int enabled = -1, grouped_enabled = 1;
    if (enabled < 0) {
        const char* e3 = getenv("B200TTS_NO_TCG");
        grouped_enabled = (e3 && atoi(e3)) ? 0 : 1;
        const char* e = getenv("B200TTS_NO_TC");
        enabled = (e && atoi(e)) ? 0 : 1;
    }
    if (!enabled || !L.allow_tc || (!L.w_tc && !L.w_tcg) || a.Tq < 128) return -1;
    if (a.act == ACT_LOGCLAMP || a.act == ACT_TANH) return -1;
    if (!(a.in_slope >= 0.f && a.in_slope <= 1.f)) return -1;   // the producers' leaky ReLU is max(x, slope * x)
    const bool needs_v3 = (a.flags & (EPI_MASK_PRE | EPI_SPLIT | EPI_ACCUM2 | EPI_GATE)) != 0;
    int dev = 0;
    if (int rc = device_once(g_tc_once, &dev, [](int d) -> int {
        B200_CUDA_OK(cudaFuncSetAttribute(tc3::conv1d_tc3_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
        B200_CUDA_OK(cudaFuncSetAttribute(tc3::conv1d_tc3s_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
        B200_CUDA_OK(cudaFuncSetAttribute(tc3::conv1d_tc3x_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
        B200_CUDA_OK(cudaFuncSetAttribute(tc3::conv1d_tc3_tf32_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
        B200_CUDA_OK(cudaFuncSetAttribute(tc3::conv1d_tc3x_tf32_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
        for (int g : {2, 4})
            for (bool x1 : {false, true})
                B200_CUDA_OK(cudaFuncSetAttribute(tc3::grouped_kernel(g, x1), cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
        int* flag = nullptr;
        B200_CUDA_OK(cudaHostAlloc((void**)&flag, sizeof(int), cudaHostAllocMapped | cudaHostAllocPortable));
        *flag = 0;
        g_tc_dev[d].err = flag;    // unified addressing: the host pointer is valid on the device
        B200_CUDA_OK(cudaDeviceGetAttribute(&g_tc_dev[d].num_sms, cudaDevAttrMultiProcessorCount, d));
        return 0;
    })) return rc;
    int* const g_tc_err = g_tc_dev[dev].err;
    const int num_sms = g_tc_dev[dev].num_sms;
    B200_REQUIRE(*reinterpret_cast<volatile int*>(g_tc_err) == 0,
                 "tcgen05 conv: an earlier launch on device %d hit a pipeline timeout (its output is invalid)", dev);
    const int rows_pad = (tc::TT + (L.K - 1) * L.dil + 7) / 8 * 8;
    // single-pass TF32 layers run the X1 twins of the same kernels.  Eligibility is always judged with the 3xTF32
    // shared-memory size, so a layer takes the same family in either mode; the launch sizes what the kernel uses.
    const bool x1 = L.tc_passes == 1;
    // ---- persistent kernel (needs 16-byte aligned activation rows for its cp.async staging; no input mask)
    const bool aligned = ((reinterpret_cast<uintptr_t>(a.x) & 15) == 0) && (a.x_cs % 4 == 0) && (a.x_bs % 4 == 0);
    const int n_rtiles = (L.Rows + L.tc_n - 1) / L.tc_n;
    const bool persistent_ok = aligned && !a.xmask &&
                               (L.ups == 1 || (!a.res && !(a.flags & EPI_ACCUM) && !a.ymask && !a.cond));
    if (grouped_enabled && persistent_ok && L.tc_grp && L.w_tcg && L.ups == 1 && !needs_v3 && !a.ymask &&
        (L.tc_grp - 1) * L.dil <= 15 && a.Tq >= 256) {
        // grouped mode of the third-generation kernel: M = tap groups x channels, N = 256 time steps, 240 per tile
        const int G = L.tc_grp, J = (L.K + G - 1) / G;
        const int rp = (tc3::TT2 + (J - 1) * G * L.dil + 7) / 8 * 8;
        if (rp <= 320 && tc3::smem_bytes3(rp, rp + 4) + 128 + tc3::GROUP_XCHG_BYTES <= 227 * 1024) {
            tc3::Tc3Args t;
            memset(&t, 0, sizeof(t));
            t.x = a.x; t.x_bs = a.x_bs; t.x_cs = a.x_cs; t.Tin = a.Tin; t.in_slope = a.in_slope;
            t.w = L.w_tcg; t.bias = L.bias; t.cond = a.cond; t.cond_bs = a.cond_bs;
            t.Cin = L.Cin; t.K = L.K; t.dil = L.dil; t.pad = L.pad; t.Rows = L.Rows; t.N = 128;
            t.KJ = J; t.dil_blk = G * L.dil; t.tstep = tc3::TSTEP_GROUPED;
            t.y = a.y; t.y_bs = a.y_bs; t.y_cs = a.y_cs; t.Tout = a.Tout; t.ups = 1; t.Tq = a.Tq;
            t.res = a.res; t.res_bs = a.res_bs; t.res_cs = a.res_cs;
            t.scale = a.scale; t.post_div = a.post_div; t.relu = (a.act == ACT_RELU); t.accum = (a.flags & EPI_ACCUM) ? 1 : 0;
            t.rows_pad = rp; t.raw_w = rp + 4;
            t.B = io.B; t.n_ttiles = (a.Tq + t.tstep - 1) / t.tstep; t.n_rtiles = 1;
            t.err = g_tc_err;
            size_t smemg = (tc3::smem_bytes3(rp, rp + 4, L.tc_passes) + 127) / 128 * 128;
            t.stage_off = (int)smemg;                          // partial-sum exchange tiles of the grouped epilogue
            smemg += tc3::GROUP_XCHG_BYTES;
            set_ragged(t, a, smemg);
            const long long tiles = (long long)t.B * t.n_ttiles;
            const int grid = (int)(tiles < num_sms ? tiles : num_sms);
            B200_CUDA_OK(launch_tc3(tc3::grouped_kernel(G, x1), grid, smemg, st, t));
            count_launch();
            dispatch_note(x1 ? DISPATCH_TC3_GROUPED_TF32 : DISPATCH_TC3_GROUPED);
            B200_CUDA_OK(cudaGetLastError());
            return 0;
        }
    }
    if (persistent_ok && L.tc_n == 128 && L.w_tc && tc3::smem_bytes3(rows_pad, rows_pad + 4) <= 227 * 1024) {
        // third generation: M = rows (128, zero padded), N = 256 time steps
        tc3::Tc3Args t;
        memset(&t, 0, sizeof(t));
        t.x = a.x; t.x_bs = a.x_bs; t.x_cs = a.x_cs; t.Tin = a.Tin; t.in_slope = a.in_slope;
        t.w = L.w_tc; t.bias = L.bias; t.cond = a.cond; t.cond_bs = a.cond_bs;
        t.Cin = L.Cin; t.K = L.K; t.dil = L.dil; t.pad = L.pad; t.Rows = L.Rows; t.N = 128;
        t.KJ = L.K; t.dil_blk = L.dil; t.tstep = tc3::TT2;
        t.y = a.y; t.y_bs = a.y_bs; t.y_cs = a.y_cs; t.Tout = a.Tout; t.ups = L.ups; t.Tq = a.Tq;
        t.res = a.res; t.res_bs = a.res_bs; t.res_cs = a.res_cs;
        t.ymask = a.ymask; t.ymask_bs = a.ymask_bs;
        t.scale = a.scale; t.post_div = a.post_div; t.relu = (a.act == ACT_RELU); t.accum = (a.flags & EPI_ACCUM) ? 1 : 0;
        t.mask_post = (a.flags & EPI_MASK_POST) ? 1 : 0;
        t.mask_pre = (a.flags & EPI_MASK_PRE) ? 1 : 0;
        t.gate = (a.flags & EPI_GATE) ? 1 : 0;
        t.split = (a.flags & EPI_SPLIT) ? a.split : 0;
        t.y2 = a.y2; t.y2_bs = a.y2_bs; t.y2_cs = a.y2_cs; t.accum2 = (a.flags & EPI_ACCUM2) ? 1 : 0;
        t.rows_pad = rows_pad; t.raw_w = rows_pad + 4;
        t.B = io.B; t.n_ttiles = (a.Tq + tc3::TT2 - 1) / tc3::TT2; t.n_rtiles = n_rtiles;
        t.err = g_tc_err;
        static int staged = -1;
        if (staged < 0) { const char* e = getenv("B200TTS_STAGED"); staged = (e && atoi(e)) ? 1 : 0; }
        size_t smem3 = tc3::smem_bytes3(rows_pad, rows_pad + 4, L.tc_passes);
        // staged (shared-memory transposed, coalesced) epilogue for K <= 3 layers.  It beat the r01 direct epilogue by 13 % on
        // those layers; since the direct epilogue prefetches without register copies (r02) the direct one wins
        // (decoder 17.2 -> 16.5 ms per bench step, same box A/B), so it is opt-in again: B200TTS_STAGED=1
        if (staged && !x1 && L.K <= 3 && L.ups == 1 && !t.gate && t.split == 0 && ((smem3 + 15) / 16 * 16 + tc3::STAGE_BYTES) <= 227 * 1024) {
            t.stage = 1;
            t.stage_off = (int)((smem3 + 15) / 16 * 16);
            smem3 = (size_t)t.stage_off + tc3::STAGE_BYTES;
        }
        // plain layers (bias, residual, accumulate): the kernel with the lean epilogue; everything else (WaveNet gate / split,
        // masks, ReLU, scale, final divide, transposed convs) the one with the general epilogue inline
        const bool plain_epi = L.ups == 1 && !t.gate && t.split == 0 && !t.relu && !t.ymask && t.scale == 1.f && t.post_div == 1.f;
        if (!t.stage && plain_epi && (smem3 + 127) / 128 * 128 + tc3::LEAN_STAGE_BYTES + tc3::ragged_table_bytes(t.B) <= 227 * 1024) {
            t.stage_off = (int)((smem3 + 127) / 128 * 128);     // per-warp transposition tiles of the lean epilogue
            smem3 = (size_t)t.stage_off + tc3::LEAN_STAGE_BYTES;
        }
        set_ragged(t, a, smem3);
        const long long tiles = (long long)t.B * t.n_ttiles * t.n_rtiles;
        const int grid = (int)(tiles < num_sms ? tiles : num_sms);
        tc3::Tc3Kernel k3 = t.stage ? tc3::conv1d_tc3s_kernel : plain_epi ? tc3::conv1d_tc3_kernel : tc3::conv1d_tc3x_kernel;
        if (x1) k3 = plain_epi ? tc3::conv1d_tc3_tf32_kernel : tc3::conv1d_tc3x_tf32_kernel;
        B200_CUDA_OK(launch_tc3(k3, grid, smem3, st, t));
        count_launch();
        dispatch_note(x1 ? DISPATCH_TC3_TF32 : t.stage ? DISPATCH_TC3_STAGED : DISPATCH_TC3);
        B200_CUDA_OK(cudaGetLastError());
        return 0;
    }
    // Everything else (fewer than 64 rows without a grouped packing, unaligned or masked inputs, shared-memory budget)
    // runs on the exact FP32-FMA kernel: the first two tcgen05 generations are no longer part of the library
    // (tools/legacy/, harness only), so a dispatch change cannot silently land on them.
    return -1;
}

int conv_tc_error_flag() {   // 1 if any tcgen05 launch (on any device) hit a pipeline timeout; call after a sync
    for (int d = 0; d < MAX_DEVICES; ++d)
        if (g_tc_dev[d].err && *reinterpret_cast<volatile int*>(g_tc_dev[d].err)) return 1;
    return 0;
}

int launch_conv(const ConvLayer& L, const ConvIO& io, cudaStream_t st) {
    B200_REQUIRE(L.w && io.x && io.y, "launch_conv: null tensor");
    ConvKArgs a;
    memset(&a, 0, sizeof(a));
    a.x = io.x; a.x_bs = io.x_bs; a.x_cs = io.x_cs; a.Tin = io.Tin;
    a.xmask = io.xmask; a.xmask_bs = io.xmask_bs; a.in_slope = io.in_slope;
    a.w = L.w; a.bias = L.bias; a.cond = io.cond; a.cond_bs = io.cond_bs;
    a.Cin = L.Cin; a.CinPad = L.CinPad; a.K = L.K; a.dil = L.dil; a.pad = L.pad; a.Rows = L.Rows; a.ups = L.ups;
    a.y = io.y; a.y_bs = io.y_bs; a.y_cs = io.y_cs; a.Tout = io.Tout;
    a.Tq = (L.ups > 1) ? (io.Tout + L.ups - 1) / L.ups : io.Tout;
    a.res = io.res; a.res_bs = io.res_bs; a.res_cs = io.res_cs;
    a.ymask = io.ymask; a.ymask_bs = io.ymask_bs;
    a.y2 = io.y2; a.y2_bs = io.y2_bs; a.y2_cs = io.y2_cs; a.split = io.split;
    a.scale = io.scale; a.post_div = io.post_div; a.act = io.act; a.act_param = io.act_param; a.flags = io.flags;
    a.lens = io.lens; a.rate_out = io.rate_out; a.need_out = io.need_out; a.rate_in = io.rate_in; a.need_in = io.need_in;
    if (a.Tq <= 0 || io.B <= 0) return 0;
    B200_REQUIRE(!(a.flags & (EPI_MASK_PRE | EPI_MASK_POST | EPI_SPLIT)) || io.ymask,
                 "launch_conv: masked/split epilogue needs ymask");
    B200_REQUIRE(!(a.flags & EPI_SPLIT) || io.y2, "launch_conv: split epilogue needs y2");
    B200_REQUIRE(!(io.ymask && L.ups > 1), "launch_conv: output mask with an upsampling layer is not supported");
    if (a.flags & EPI_GATE) {
        B200_REQUIRE(L.ups == 1 && !io.res && a.act == ACT_NONE, "launch_conv: gate epilogue takes no other options");
        if (int rc = try_launch_tc(L, io, a, st); rc != -1) return rc;
        return launch_cic<KEPI_GATE>(a, L.co_tile, io.B, L.RowsPad, st);
    }
    if (a.act == ACT_TANH) {
        B200_REQUIRE(L.ups == 1 && !io.res && !io.cond && a.flags == 0 && a.scale == 1.f && a.post_div == 1.f,
                     "launch_conv: tanh epilogue takes no other options");
        // conv_post (one output row, 7 taps): streaming kernel when rows are 16-byte aligned
        if (L.Rows == 1 && L.K == 7 && L.dil == 1 && L.pad == 3 && !a.xmask && a.Tin == a.Tout && (a.Tout % 4) == 0 &&
            (a.x_cs % 4) == 0 && (a.x_bs % 4) == 0 && (a.y_bs % 4) == 0 && (reinterpret_cast<uintptr_t>(a.x) & 15) == 0 &&
            (reinterpret_cast<uintptr_t>(a.y) & 15) == 0 && (size_t)L.Cin * L.K * 4 <= 48 * 1024) {
            dim3 grid((a.Tout / 4 + 255) / 256, io.B);
            if (grid.y <= 65535) {
                conv1d_row1_kernel<7><<<grid, 256, (size_t)L.Cin * L.K * 4, st>>>(a.x, a.x_bs, a.x_cs, L.Cin, a.Tout, L.w,
                                                                                 L.co_tile, L.bias, a.in_slope, a.act, a.y,
                                                                                 a.y_bs, io.peak_bits, a.lens, a.rate_out,
                                                                                 a.need_out, a.need_in);
                count_launch();
                dispatch_note(DISPATCH_ROW1);
                B200_CUDA_OK(cudaGetLastError());
                return 0;
            }
        }
        if (int rc = launch_cic<KEPI_TANH>(a, L.co_tile, io.B, L.RowsPad, st)) return rc;
        if (io.peak_bits) {   // the streaming kernel was not eligible: fold the peak in a pass of its own
            B200_REQUIRE(a.y_cs == a.Tout && a.y_bs == (long long)L.Rows * a.Tout, "launch_conv: peak needs a dense output");
            return launch_absmax(a.y, (long long)io.B * L.Rows * a.Tout, io.peak_bits, st);
        }
        return 0;
    }
    if (int rc = try_launch_tc(L, io, a, st); rc != -1) return rc;
    const bool plain = L.ups == 1 && !io.res && a.scale == 1.f && a.post_div == 1.f &&
                       (a.flags & ~(EPI_MASK_POST | EPI_MASK_PRE)) == 0;
    if (plain) return launch_cic<KEPI_PLAIN>(a, L.co_tile, io.B, L.RowsPad, st);
    B200_REQUIRE(a.act != ACT_LOGCLAMP, "launch_conv: log-clamp activation only with the plain epilogue");
    return launch_cic<KEPI_GENERIC>(a, L.co_tile, io.B, L.RowsPad, st);
}

}  // namespace b200tts
