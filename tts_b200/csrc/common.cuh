// tts_b200 -- shared declarations for the sm_100a hot-path kernels.
// Host-side C++ here is the "engine" above the kernels; the only public surface is the
// C ABI in include/tts_b200.h (implemented in capi.cu).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <atomic>
#include <mutex>
#include <string>
#include <vector>

namespace b200tts {

// ------------------------------------------------------------------ errors
void set_error(const char* fmt, ...);
const char* last_error();

#define B200_CUDA_OK(expr)                                                                  \
    do {                                                                                    \
        cudaError_t _e = (expr);                                                            \
        if (_e != cudaSuccess) {                                                            \
            ::b200tts::set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #expr,              \
                                 cudaGetErrorString(_e));                                   \
            return 2;                                                                       \
        }                                                                                   \
    } while (0)

#define B200_REQUIRE(cond, ...)                                                             \
    do {                                                                                    \
        if (!(cond)) {                                                                      \
            ::b200tts::set_error(__VA_ARGS__);                                              \
            return 1;                                                                       \
        }                                                                                   \
    } while (0)

// ------------------------------------------------------------------ per-device one-time initialisation
// Function attributes (cudaFuncSetAttribute), device-side flags and the SM count belong to ONE device; the Python
// layer picks the device per tensor, so "done once per process" would leave a second GPU of the same process
// unconfigured.  State is keyed by cudaGetDevice() and set up under a mutex (handles may be shared across threads).
constexpr int MAX_DEVICES = 64;
struct DeviceOnce {
    std::mutex mu;
    std::atomic<bool> done[MAX_DEVICES];
    DeviceOnce() { for (auto& d : done) d.store(false); }
};
// Runs f(device) the first time it is called with a given current device; returns f's status (0 = ok) or 2.
template <class F>
inline int device_once(DeviceOnce& o, int* dev_out, F&& f) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= MAX_DEVICES) {
        set_error("device_once: cannot identify the current CUDA device");
        return 2;
    }
    if (dev_out) *dev_out = dev;
    if (o.done[dev].load(std::memory_order_acquire)) return 0;
    std::lock_guard<std::mutex> g(o.mu);
    if (o.done[dev].load(std::memory_order_relaxed)) return 0;
    if (int rc = f(dev)) return rc;
    o.done[dev].store(true, std::memory_order_release);
    return 0;
}

// launch accounting (bench.py reports "gpu_launches" from this counter)
extern unsigned long long g_launch_count;
inline void count_launch(int n = 1) { g_launch_count += (unsigned long long)n; }

// ------------------------------------------------------------------ conv1d implicit GEMM
// y[b, row, t] = epilogue( sum_ci sum_k W[row, ci, k] * prologue(x[b, ci, t + k*dil - pad]) )
//
// prologue : x *= xmask[b,t] (optional);  x = leaky_relu(x, in_slope)  (1.0 = identity)
// epilogue : v = acc + bias[row] + cond[b,row]
//            GATE      : rows come in (tanh,sigmoid) pairs -> v = tanh(v0)*sigmoid(v1), one output row per pair
//            act       : 0 none, 1 relu, 2 tanh
//            mask_pre  : v *= ymask[b,t]
//            res       : v += res[b,row,t]
//            scale     : v *= scale
//            accum     : v += y_old
//            post_div  : v /= post_div
//            mask_post : v *= ymask[b,t]
//            SPLIT (WN res/skip): rows <  split -> (y , accum=1, mask_post=1)
//                                 rows >= split -> (y2, accum=accum2, no mask), row index -= split
//            ups > 1 (polyphase transposed conv): row r -> channel r/ups, time q*ups + r%ups
enum : int { ACT_NONE = 0, ACT_RELU = 1, ACT_TANH = 2, ACT_LOGCLAMP = 3 };  // LOGCLAMP: log(max(v, act_param))
enum : int { EPI_GATE = 1, EPI_MASK_PRE = 2, EPI_MASK_POST = 4, EPI_ACCUM = 8, EPI_SPLIT = 16, EPI_ACCUM2 = 32 };

struct ConvLayer {            // immutable after pack(); owned by an engine handle
    float* w = nullptr;       // device, packed [row_tiles][CinPad][K][CO_T]
    float* bias = nullptr;    // device, [RowsPad] (zeros when the layer has no bias)
    int Cin = 0, CinPad = 0;  // input channels (padded to the ci chunk)
    int Rows = 0, RowsPad = 0;  // GEMM rows (Cout, or Cout*ups for transposed conv; 2*H interleaved for gate)
    int K = 1, dil = 1, pad = 0;
    int ups = 1;              // >1: polyphase ConvTranspose1d
    int co_tile = 64;         // 32 or 64
    int tr_kernel = 0, tr_pad = 0;  // original transposed-conv kernel size / padding (for Tout)
    float* w_tc = nullptr;    // device, tcgen05 packing [n_tile][chunk][tap]{hi,lo}[slab][N][4] (null: layer not eligible)
    int tc_n = 0;             // columns (output rows) per tcgen05 CTA
    float* w_tcg = nullptr;   // device, grouped tcgen05 packing [chunk][tap block]{hi,lo}[slab][128][4] (rows == 32 / 64)
    int tc_grp = 0;           // tap groups of the grouped packing (128 / rows), 0: none
    bool allow_tc = false;    // engines opt layers into the 3xTF32 tensor-core path (decoder / flow); the text and
                              // duration path stays on the exact FP32 FMA kernel so durations remain bit-stable
    int tc_passes = 3;        // how w_tc / w_tcg were packed: 3 (3xTF32, {hi,lo}) or 1 (single-pass TF32, rounded to
                              // nearest); selects the matching tcgen05 kernels.  The FP32-FMA / single-row kernels ignore it
};

struct ConvIO {
    const float* x = nullptr; long long x_bs = 0; int x_cs = 0; int Tin = 0;
    const float* xmask = nullptr; long long xmask_bs = 0;
    float in_slope = 1.0f;
    const float* cond = nullptr; long long cond_bs = 0;   // [B, RowsPad-compatible] per-(b,row) bias
    float* y = nullptr; long long y_bs = 0; int y_cs = 0; int Tout = 0;
    const float* res = nullptr; long long res_bs = 0; int res_cs = 0;
    const float* ymask = nullptr; long long ymask_bs = 0;
    float* y2 = nullptr; long long y2_bs = 0; int y2_cs = 0;
    int split = 0;
    float scale = 1.0f;
    float post_div = 1.0f;   // applied after accumulation (MRF mean: z_sum / num_kernels)
    int act = ACT_NONE;
    float act_param = 0.f;
    int flags = 0;
    int B = 1;
    unsigned* peak_bits = nullptr;   // single-row tanh kernel only: atomicMax of |y| (as float bits) over everything stored
    // ragged batch (null: dense).  lens[b] = valid FRAMES of row b; this launch's output is only computed below
    // lens[b] * rate_out + need_out (time steps of y; for a transposed conv `rate_out` counts GEMM columns, i.e. input
    // steps), its input is read as zero from lens[b] * rate_in + need_in on.  Honoured by the persistent tcgen05 kernels
    // and the single-row kernel; the FMA tile kernel computes the full tensor (valid samples are identical either way).
    const int* lens = nullptr; int rate_out = 1, need_out = 0, rate_in = 1, need_in = 0;
};

// Host weights in PyTorch layout.  conv: w[Cout][Cin][K];  transposed: w[Cin][Cout][Kt].
// gate_half > 0 interleaves rows (p, p+gate_half) for the fused WaveNet gate.
// in_perm / out_perm (nullable) remap logical->physical channels (flow channel flips).
// tc_passes: 3 (3xTF32) or 1 (single-pass TF32) for the tensor-core packings, see ConvLayer::tc_passes.
int pack_conv(ConvLayer& L, const float* w, const float* bias, int Cout, int Cin, int K, int dil, int pad,
              int gate_half = 0, const int* in_perm = nullptr, const int* out_perm = nullptr, int tc_passes = 3);
int pack_conv_transpose(ConvLayer& L, const float* w, const float* bias, int Cin, int Cout, int Kt, int stride,
                        int padding, int tc_passes = 3);
void free_conv(ConvLayer& L);
int launch_conv(const ConvLayer& L, const ConvIO& io, cudaStream_t stream);
int conv_tc_error_flag();
// which kernel family a launch_conv call dispatched to (recorded per thread between dispatch_begin/end; tests pin it)
enum : int { DISPATCH_FMA = 0, DISPATCH_TC1 = 1, DISPATCH_TC2 = 2, DISPATCH_TC3 = 3, DISPATCH_TC3_STAGED = 4,
             DISPATCH_TC3_GROUPED = 5, DISPATCH_ROW1 = 6, DISPATCH_RESBLOCK = 7, DISPATCH_TC3_TF32 = 8,
             DISPATCH_TC3_GROUPED_TF32 = 9 };
void dispatch_begin();
int dispatch_end(int* ids, int cap);
void dispatch_note(int id);
inline int conv_transpose_out_len(const ConvLayer& L, int Tin) {
    return (Tin - 1) * L.ups - 2 * L.tr_pad + L.tr_kernel;
}

// small helpers shared by the engines
int upload(float** dst, const float* src, size_t n);   // cudaMalloc + H2D copy

// ------------------------------------------------------------------ bump allocator over a caller workspace
struct Arena {
    char* base; size_t cap; size_t off;
    Arena(void* p, size_t bytes) : base((char*)p), cap(bytes), off(0) {}
    float* f32(size_t n) {
        size_t bytes = (n * sizeof(float) + 255) & ~size_t(255);
        if (off + bytes > cap) return nullptr;
        float* r = (float*)(base + off);
        off += bytes;
        return r;
    }
};
inline size_t arena_bytes(size_t n_floats) { return (n_floats * sizeof(float) + 255) & ~size_t(255); }

}  // namespace b200tts
