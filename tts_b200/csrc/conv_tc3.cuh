// Persistent tcgen05 3xTF32 conv1d, third generation: M = output rows (weights are the A operand), N = 256 time
// steps (the activation window is the B operand), D[row, t] in TMEM (128 lanes x 256 columns, double buffered).
//
// Why this orientation: measured on B200 (profiles/r01_tc_notes.md) an SS-mode tcgen05.mma with M = 128 costs ~135
// cycles whatever N is -- the 128-row A operand streams from shared memory at about one 32-byte row per clock.  With
// the time axis as N = 256 each instruction carries 128 x 256 x 8 MACs in those ~128 cycles instead of 128 x N_cout x 8.
// The activation tile keeps the row-shift property (rows are 16 B apart), so tap k is still just a descriptor
// start-address offset of k*dil rows -- now on the B operand.
//
//   warps 0-3, 12-15 epilogue  : two column halves x four TMEM lane quarters.  Plain layers: lean path (TMEM -> + bias ->
//                                per-warp shared tile -> 8 rows x 64 B global accesses, residual / accumulate loads in that
//                                mapping one group ahead); everything else: the general path (gate, split, masks, polyphase)
//   warps 4-9        producers : cp.async raw [8 ch][time] windows (4-deep ring) -> leaky-ReLU + hi/lo split -> K-major slabs
//                                (5 stages)
//   warp  10         loader    : per-tap weight blocks {hi,lo}[2 slabs][128 rows][4] by cp.async.bulk, one lane per ring slot
//                                (6 slots; r02 sweep in profiles/r02_epilogue_instruction_bound.md: 5 activation stages + 6
//                                weight slots beat 3 + 10 by ~3 %)
//   warp  11         MMA       : converged warp, one elected lane issues 3 tcgen05.mma (lo*hi, hi*lo, hi*hi) per tap and
//                                chunk and commits to mbarriers
//
// Single-pass TF32 mode (template flag X1, the opt-in `tf32` precision of the HiFiGAN decoder): the producers round the
// activation to TF32 (cvt.rna: nearest, ties away from zero) instead of splitting it, the packer rounds the weights with
// the same rule, there are no lo slabs (half the activation stage, 4 KB tap blocks) and one MMA per tap.  Everything
// else -- schedule, barriers, partial-tile N, epilogues -- is the same code.
//
// Grouped mode (GRP = 2 / 4) for narrow layers (exactly 64 / 32 output rows, the last two HiFiGAN stages): the 128
// MMA rows are GRP tap-groups x (128/GRP) channels -- row g * (128/GRP) + c carries the weights of channel c for taps
// g, g+GRP, g+2*GRP, ... so one instruction stream of ceil(K/GRP) "tap blocks" (B shifted by GRP*dil rows per block)
// replaces K of them and no MMA row is zero padding.  D_g[c, col] then still misses its own g*dil shift; a TMEM lane
// quarter holds one group, so each epilogue warp applies the shift as the column offset of its tcgen05.ld and the four
// warps of a column half sum their partials through a shared tile.  Tiles advance by 240 columns so every shifted read
// stays inside the 256-column accumulator.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <type_traits>

#include "conv_tc.cuh"   // descriptor / barrier helpers

namespace b200tts {
namespace tc3 {

using namespace tc;       // smem_u32, mbar_*, make_desc, make_idesc, mma_tf32, mma_commit, tmem_ld16, fences

constexpr int TT2 = 256;          // time steps per tile = MMA N
constexpr int MROWS = 128;        // output rows per tile = MMA M (weight rows are zero padded up to it)
constexpr int KC2 = 8;            // input channels per chunk (2 slabs, one MMA k-step)
constexpr int RAWS = 324;         // raw (cp.async) row stride in floats: the widest window (320 slab rows + 4), a constant so
                                  // that the transform's shared loads use immediate offsets
#ifndef TC3_NRAW
#define TC3_NRAW 4
#endif
#ifndef TC3_NA2
#define TC3_NA2 5
#endif
#ifndef TC3_NB2
#define TC3_NB2 6
#endif
constexpr int NRAW = TC3_NRAW;    // raw (cp.async) ring depth
constexpr int NA2 = TC3_NA2;      // transformed activation stages
constexpr int NB2 = TC3_NB2;      // weight ring depth (one tap block per slot: 8 KB, 4 KB single-pass)
#ifndef TC3_RDEPTH
#define TC3_RDEPTH 2
#endif
#ifndef TC3_NPW
#define TC3_NPW 6
#endif
constexpr int NPW = TC3_NPW;      // producer warps.  r02: a producer warp spends ~400 dependent instructions per chunk (~2000
                                  // cycles) and four of them paced every K <= 7 layer; eight halve the per-warp share
constexpr int NPROD = 32 * NPW;
constexpr int W_PROD = 4, W_LOAD = 4 + NPW, W_MMA = 5 + NPW, W_EPI2 = 6 + NPW;   // warp roles: 0-3 and W_EPI2..+3 epilogue
constexpr int NTHREADS2 = 32 * (W_EPI2 + 4);

struct Tc3Args {
    const float* x; long long x_bs; int x_cs; int Tin;
    float in_slope;
    const float* w;            // packed [row_tile][chunk][tap]{hi[2][128][4], lo[2][128][4]} (single pass: {w[2][128][4]})
    const float* bias;
    const float* cond; long long cond_bs;
    int Cin, K, dil, pad, Rows, N;
    float* y; long long y_bs; int y_cs; int Tout;
    int ups;                   // 1, or the polyphase factor of a transposed conv (row r -> channel r/ups, phase r%ups)
    int Tq;                    // GEMM columns in time (= Tout for ups == 1)
    const float* res; long long res_bs; int res_cs;
    const float* ymask; long long ymask_bs;
    float scale; float post_div; int relu; int accum; int mask_post;
    int mask_pre;              // multiply by ymask before the residual / accumulate (coupling `post`)
    int gate;                  // rows are (tanh, sigmoid) pairs: out[r/2] = tanh(v[2p]) * sigmoid(v[2p+1])  (WaveNet)
    int split;                 // > 0: rows < split -> y (accumulate, mask); rows >= split -> y2 (accumulate iff accum2)
    float* y2; long long y2_bs; int y2_cs; int accum2;
    int KJ;                    // tap blocks per chunk (= K, or ceil(K / GRP) in grouped mode)
    int dil_blk;               // B-row shift between tap blocks (= dil, or GRP * dil)
    int tstep;                 // time steps a tile advances (= TT2, or 240 in grouped mode)
    int rows_pad;              // slab rows  (TT2 + halo, multiple of 8)
    int raw_w;                 // raw row width in floats (rows_pad + 4, multiple of 4)
    int B, n_ttiles, n_rtiles;
    int* err;
    unsigned long long* trace;  // optional [grid][32] globaltimer stamps (debug)
    int stage;                  // != 0: wide-layer epilogue goes through per-warp shared tiles (coalesced global access)
    int stage_off;              // byte offset of those tiles in dynamic shared memory (8 warps x 5120 B); grouped mode:
                                // offset of the GROUP_XCHG_BYTES partial-sum exchange tiles
    int dbg;                    // harness-only bottleneck probes: 1 no cp.async, 2 no transform, 4 no epilogue loads, 8 no stores, 16 no MMA, 32 epilogue = handshake only, 64 no test_wait probe, 128 lane = row lean epilogue,
                                // 512 full-width MMAs on partial tiles, 256 (with 16) the MMA warp arrives on its barriers itself instead of tcgen05.commit (racecheck probe)
    // ---- ragged batches (null lens: every row spans the full tensor).  Row b only has tiles for GEMM columns below
    // min(Tq, lens[b] * rate_q + need_q) and its input is read as zero from min(Tin, lens[b] * rate_in + need_in) on:
    // padded frames cost nothing, and `need` keeps every sample below lens[b] bit-identical to the full computation
    // (it is the receptive field of the layers that still follow, worked out per launch by the engine).
    const int* lens; int rate_q, need_q, rate_in, need_in;
    int pref_off;               // byte offset in dynamic shared memory of the (B + 1)-entry tile prefix table
};

// passes: 3 (3xTF32, {hi,lo} slabs) or 1 (single-pass TF32, one slab pair per activation stage and weight block)
static inline size_t smem_bytes3(int rows_pad, int raw_w, int passes = 3) {
    (void)raw_w;     // raw rows are stored at the fixed stride RAWS
    const size_t slabs = passes == 1 ? 2 : 4;
    return (size_t)NRAW * KC2 * RAWS * 4 + (size_t)NA2 * (slabs * rows_pad * 16) + (size_t)NB2 * (slabs * MROWS * 16) + 512;
}
static inline size_t ragged_table_bytes(int B) { return ((size_t)(B + 1) * sizeof(int) + 15) / 16 * 16; }

__device__ __forceinline__ void cp_async16(uint32_t dst, const void* src) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async16_zfill(uint32_t dst, const void* src, uint32_t src_bytes) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(src_bytes) : "memory");
}
// tcgen05.ld without the wait: issue several, then one tmem_wait_ld() (the loads' latencies overlap)
__device__ __forceinline__ void tmem_ld16_nowait(uint32_t taddr, uint32_t* r) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
                   "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
                 : "r"(taddr));
}
template <int N>
__device__ __forceinline__ void tmem_ld_nowait(uint32_t taddr, uint32_t* r) {   // N = 1, 2, 4, 8 or 16 columns
    if constexpr (N == 16) tmem_ld16_nowait(taddr, r);
    else if constexpr (N == 8)
        asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                     : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]) : "r"(taddr));
    else if constexpr (N == 4)
        asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0,%1,%2,%3}, [%4];" : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(taddr));
    else if constexpr (N == 2)
        asm volatile("tcgen05.ld.sync.aligned.32x32b.x2.b32 {%0,%1}, [%2];" : "=r"(r[0]), "=r"(r[1]) : "r"(taddr));
    else
        asm volatile("tcgen05.ld.sync.aligned.32x32b.x1.b32 {%0}, [%1];" : "=r"(r[0]) : "r"(taddr));
}
// 16 columns x 32 lanes of zeros into TMEM (kernel start: stale accumulator columns must at least be finite, see the MMA warp)
__device__ __forceinline__ void tmem_st16_zero(uint32_t taddr) {
    const uint32_t z = 0u;
    asm volatile("tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1,%1,%1,%1,%1,%1,%1,%1,%1,%1,%1,%1,%1,%1,%1,%1};" ::"r"(taddr), "r"(z) : "memory");
}
// round to TF32, nearest with ties away from zero (the packer's host rounding, conv1d.cu tf32_rna, is the same rule)
__device__ __forceinline__ float tf32_rna(float x) {
    uint32_t r;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
    return __uint_as_float(r);
}
__device__ __forceinline__ void tmem_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void named_bar_sync(int id, int n) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(n) : "memory"); }

#define TC3_STAMP(slot) do { if (a.trace) a.trace[(size_t)blockIdx.x * 32 + (slot)] = gtime(); } while (0)

constexpr int STAGE_BYTES = 8 * 5120;   // staged epilogue: per epilogue warp an output and a residual tile of [32][20] floats
constexpr int TSTEP_GROUPED = 240;   // 15 chunks of 16 columns: leaves room for the (GRP-1)*dil <= 15 column shift

// Lean epilogue of one interior tile half (plain layers: bias, optional residual HR / accumulate HA): lane = one output row
// (padding lanes were clamped to the last real row, so their loads are harmless and only their stores are predicated),
// 128 columns in steps of NC.  HR / HA are compile-time so that every load is an UNCONDITIONAL definition: with `if (hr) ld`
// ptxas kept the prefetched sets in local memory (store right after the load = wait for it), which serialised the steps
// (r02 ncu source view: 86 % of the epilogue samples).  Software pipeline: the TMEM load and the residual / accumulate
// loads of step g+1 fly while step g is finished.  Same operations in the same order as the general code (bit-identical).
template <bool HR, bool HA>
__device__ __forceinline__ void lean_rows(uint32_t dbase, float bias, const float* rp, float* yp, bool st_ok) {
    constexpr int NC = 8;                      // columns per step (two float4 = one 32-byte sector per row)
    uint32_t vA[NC], vB[NC];
    float rA[NC], oA[NC], rB[NC], oB[NC];
    auto pf = [&](int cg, float* r_, float* o_) {
#pragma unroll
        for (int j = 0; j < NC / 4; ++j) {
            if constexpr (HR) asm volatile("ld.global.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(r_[4 * j]), "=f"(r_[4 * j + 1]), "=f"(r_[4 * j + 2]), "=f"(r_[4 * j + 3]) : "l"(rp + cg + 4 * j));
            if constexpr (HA) asm volatile("ld.global.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(o_[4 * j]), "=f"(o_[4 * j + 1]), "=f"(o_[4 * j + 2]), "=f"(o_[4 * j + 3]) : "l"(yp + cg + 4 * j));
        }
    };
    auto fin = [&](int cg, const uint32_t* v, const float* rv, const float* ov) {
        float u[NC];
#pragma unroll
        for (int i = 0; i < NC; ++i) {
            float t = __uint_as_float(v[i]) + bias;
            if constexpr (HR) t += rv[i];
            if constexpr (HA) t += ov[i];
            u[i] = t;
        }
        if (st_ok) {
#pragma unroll
            for (int j = 0; j < NC / 4; ++j)
                *reinterpret_cast<float4*>(yp + cg + 4 * j) = make_float4(u[4 * j], u[4 * j + 1], u[4 * j + 2], u[4 * j + 3]);
        }
    };
    pf(0, rA, oA);
    tmem_ld_nowait<NC>(dbase, vA);
#pragma unroll 1
    for (int cg = 0; cg < 128; cg += 2 * NC) {
        pf(cg + NC, rB, oB);
        tmem_wait_ld();
        tmem_ld_nowait<NC>(dbase + (uint32_t)(cg + NC), vB);
        fin(cg, vA, rA, oA);
        if (cg + 2 * NC < 128) pf(cg + 2 * NC, rA, oA);
        tmem_wait_ld();
        if (cg + 2 * NC < 128) tmem_ld_nowait<NC>(dbase + (uint32_t)(cg + 2 * NC), vA);
        fin(cg + NC, vB, rB, oB);
    }
}

// Lean epilogue, transposing variant (the default when its 20 KB of shared memory fit).  With lane = row every float4
// LDG / STG of lean_rows touches 32 different 128-byte lines; r02 ablation: with the epilogue's global accesses switched
// off the K = 3 layers ran 1.7x faster although the epilogue was not the pacing role -- its 32-wavefront instructions
// stall the producers' copies in the shared LSU pipe.  Here a warp's 32 x 16 block goes through a private padded shared
// tile once, so that lane (r8 = lane & 7, p4 = lane >> 3) owns float4 p4 of rows 8 i + r8: every global instruction covers
// 8 rows x 64 contiguous bytes (4x fewer wavefronts, whole sectors), the residual / accumulate loads go straight to
// registers in that mapping (no second tile).  ((acc + bias) + res) + old, as in the general code: bit-identical.
constexpr int LEAN_TILE_FLOATS = 32 * 20;                 // per epilogue warp: [32 rows][16 + 4 pad] floats (conflict-free both ways)
constexpr int LEAN_STAGE_BYTES = 8 * LEAN_TILE_FLOATS * 4;
template <bool HR, bool HA>
__device__ __forceinline__ void lean_rows_t(uint32_t dbase, float bias, float* tO, int lane, const float* rq, float* yq,
                                            long long rcs, long long ycs, int row0, int Rows, bool do_st) {
    const int r8 = lane & 7, p4 = lane >> 3;
    const float* rrow[4];
    float* yrow[4];
    bool st_ok[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int ri = row0 + 8 * i + r8, rci = ri < Rows ? ri : Rows - 1;       // padding rows: loads clamped, stores off
        rrow[i] = rq + (long long)rci * rcs + 4 * p4;
        yrow[i] = yq + (long long)rci * ycs + 4 * p4;
        st_ok[i] = do_st && ri < Rows;
    }
    float* tw = tO + lane * 20;                          // lane = row view
    const float* tr = tO + r8 * 20 + 4 * p4;             // (r8, p4) view, + i * 160
    constexpr int D = TC3_RDEPTH;                        // residual register sets: loads run D - 1 column groups ahead
    float r0[16], r1[16], r2[D == 4 ? 16 : 1], r3[D == 4 ? 16 : 1];
    static_assert(D == 2 || D == 4, "TC3_RDEPTH must be 2 or 4");
    auto pf = [&](int cg, float* r_) {
        if constexpr (HR) {
#pragma unroll
            for (int i = 0; i < 4; ++i)
                asm volatile("ld.global.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(r_[4 * i]), "=f"(r_[4 * i + 1]), "=f"(r_[4 * i + 2]), "=f"(r_[4 * i + 3]) : "l"(rrow[i] + cg));
        }
    };
    auto group = [&](int cg, const float* rv, float* rn) {
        float o[16];
        if (cg + 16 * (D - 1) < 128) pf(cg + 16 * (D - 1), rn);
        if constexpr (HA) {
#pragma unroll
            for (int i = 0; i < 4; ++i)
                asm volatile("ld.global.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(o[4 * i]), "=f"(o[4 * i + 1]), "=f"(o[4 * i + 2]), "=f"(o[4 * i + 3]) : "l"(yrow[i] + cg));
        }
        uint32_t v[16];
        tmem_ld16_nowait(dbase + (uint32_t)cg, v);
        tmem_wait_ld();
#pragma unroll
        for (int j = 0; j < 4; ++j)
            *reinterpret_cast<float4*>(tw + 4 * j) = make_float4(__uint_as_float(v[4 * j]) + bias, __uint_as_float(v[4 * j + 1]) + bias,
                                                                 __uint_as_float(v[4 * j + 2]) + bias, __uint_as_float(v[4 * j + 3]) + bias);
        __syncwarp();
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            float4 t = *reinterpret_cast<const float4*>(tr + i * 160);
            if constexpr (HR) { t.x += rv[4 * i]; t.y += rv[4 * i + 1]; t.z += rv[4 * i + 2]; t.w += rv[4 * i + 3]; }
            if constexpr (HA) { t.x += o[4 * i]; t.y += o[4 * i + 1]; t.z += o[4 * i + 2]; t.w += o[4 * i + 3]; }
            if (st_ok[i]) *reinterpret_cast<float4*>(yrow[i] + cg) = t;
        }
        __syncwarp();
    };
    if constexpr (D == 2) {
        pf(0, r0);
#pragma unroll 1
        for (int cg = 0; cg < 128; cg += 32) {
            group(cg, r0, r1);
            group(cg + 16, r1, r0);
        }
    } else {
        pf(0, r0); pf(16, r1); pf(32, r2);
#pragma unroll 1
        for (int cg = 0; cg < 128; cg += 64) {
            group(cg, r0, r3);
            group(cg + 16, r1, r0);
            group(cg + 32, r2, r1);
            group(cg + 48, r3, r2);
        }
    }
}

// Everything the lean epilogue does not cover (WaveNet gate / res-skip split, masks, ReLU, scale, final divide, polyphase
// stores of the transposed convs, edge tiles): one tile half per call.  Deliberately NOT inlined: inside the tile loop its
// loop invariants were hoisted across the lean path and pushed that path's prefetched values out of registers.
template <bool STAGED>
__device__ __forceinline__ void general_tile_body(const Tc3Args& a, unsigned char* smem, uint32_t tmem_base, uint32_t acc_cols,
                                                  int b, int rt, int q0, int buf, int lq, int half, int lane, int warp) {
    const int ups = a.ups;
    const int r = rt * MROWS + lq * 32 + lane;             // GEMM row of this lane
    const bool rok = r < a.Rows;
    const int rc = rok ? r : a.Rows - 1;
    const uint32_t dbase = tmem_base + (uint32_t)buf * acc_cols + ((uint32_t)(lq * 32) << 16) + (uint32_t)(half * 128);
    const int qb = q0 + half * 128;
    float bias = a.bias[rc];
    if (a.cond) bias += __ldg(a.cond + (long long)b * a.cond_bs + rc);
    if (a.gate) {
        // WaveNet gate (wavenet.py:6-13): even lane = tanh argument, odd lane = sigmoid argument of row r/2
        float* yrow = a.y + (long long)b * a.y_bs + (long long)(rc >> 1) * a.y_cs;
        const bool vec_ok = ((a.y_cs & 3) == 0) && ((reinterpret_cast<uintptr_t>(yrow) & 15) == 0);
        const bool even = (lane & 1) == 0;
        for (int cg = 0; cg < 128; cg += 16) {
            float v[16];
            tmem_ld16(dbase + (uint32_t)cg, v);
            const int q = qb + cg;
#pragma unroll
            for (int i = 0; i < 16; ++i) {
                const float u = v[i] + bias;
                const float act = even ? tanhf(u) : 1.f / (1.f + expf(-u));
                const float other = __shfl_xor_sync(0xffffffffu, act, 1);
                v[i] = act * other;
            }
            if (rok && even) {
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const int qq = q + 4 * j;
                    if (vec_ok && qq + 3 < a.Tout) *reinterpret_cast<float4*>(yrow + qq) = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
                    else {
#pragma unroll
                        for (int e = 0; e < 4; ++e) if (qq + e < a.Tout) yrow[qq + e] = v[4 * j + e];
                    }
                }
            }
        }
    } else if (STAGED && ups == 1 && a.stage && a.split == 0 && qb + 128 <= a.Tout && ((a.y_cs | a.y_bs) & 3) == 0 &&
               (reinterpret_cast<uintptr_t>(a.y) & 15) == 0 &&
               (!a.res || ((((a.res_cs | a.res_bs) & 3) == 0) && (reinterpret_cast<uintptr_t>(a.res) & 15) == 0))) {
        // ---- staged epilogue (interior tiles of wide layers).  With lane = row every float4 LDG / STG of the
        // direct path touches 32 different cache lines; measured, that L1 wavefront time is not hidden
        // (profiles/r01_tc_grouped_notes.md).  Here each warp transposes its 32 x 16 block through a private
        // shared tile: global accesses are 8 rows x 64 contiguous bytes per instruction (4x fewer wavefronts),
        // the residual arrives by cp.async one column group ahead.
        const int ew = (warp < 4) ? warp : warp - W_EPI2 + 4;                       // epilogue warp 0..7
        float* tO = reinterpret_cast<float*>(smem + a.stage_off) + ew * 1280;   // [32][20]
        float* tR = tO + 640;
        const int r8 = lane & 7, p4 = lane >> 3;
        const int Rbase = rt * MROWS + lq * 32 + r8;                        // + 8*i
        float* ybase = a.y + (long long)b * a.y_bs + (long long)Rbase * a.y_cs + qb + 4 * p4;
        const float* rbase = (a.res && !(a.dbg & 4)) ? a.res + (long long)b * a.res_bs + (long long)Rbase * a.res_cs + qb + 4 * p4 : nullptr;
        const bool acc_r = a.accum != 0 && !(a.dbg & 4), mpost_r = a.mask_post != 0, do_store = !(a.dbg & 8);
        const float* mrow = a.ymask ? a.ymask + (long long)b * a.ymask_bs : nullptr;
        float* yrow = a.y + (long long)b * a.y_bs + (long long)rc * a.y_cs;   // lane = row view (accumulate loads)
        auto issue_res = [&](int cg) {
            if (!rbase) return;
#pragma unroll
            for (int i = 0; i < 4; ++i)
                if (Rbase + 8 * i < a.Rows)
                    cp_async16_zfill(smem_u32(tR + (8 * i + r8) * 20 + 4 * p4), rbase + (long long)(8 * i) * a.res_cs + cg, 16u);
            asm volatile("cp.async.commit_group;" ::: "memory");
        };
        auto prefetch_acc = [&](int cg, float* o_) {
            if (!acc_r || !rok) return;
#pragma unroll
            for (int j = 0; j < 4; ++j)
                asm volatile("ld.global.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(o_[4 * j]), "=f"(o_[4 * j + 1]), "=f"(o_[4 * j + 2]), "=f"(o_[4 * j + 3]) : "l"(yrow + qb + cg + 4 * j));
        };
        issue_res(0);
#pragma unroll 1
        for (int cg = 0; cg < 128; cg += 16) {
            float v[16], ov[16], rv[16];
            prefetch_acc(cg, ov);           // accumulate-into-destination (two layers per stage): same-group load
            if (rbase) {
                asm volatile("cp.async.wait_group 0;" ::: "memory");
                __syncwarp();
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const float4 t4 = *reinterpret_cast<const float4*>(tR + lane * 20 + 4 * j);
                    rv[4 * j] = t4.x; rv[4 * j + 1] = t4.y; rv[4 * j + 2] = t4.z; rv[4 * j + 3] = t4.w;
                }
                __syncwarp();
                if (cg + 16 < 128) issue_res(cg + 16);
            }
            tmem_ld16(dbase + (uint32_t)cg, v);
            const int q = qb + cg;
#pragma unroll
            for (int i = 0; i < 16; ++i) {
                float u = v[i] + bias;
                if (a.relu) u = fmaxf(u, 0.f);
                const float mk = mrow ? __ldg(mrow + q + i) : 1.f;
                if (a.mask_pre) u *= mk;
                if (rbase) u += rv[i];
                u *= a.scale;
                if (acc_r) u += ov[i];
                if (a.post_div != 1.f) u = u / a.post_div;
                if (mpost_r) u *= mk;
                v[i] = u;
            }
#pragma unroll
            for (int j = 0; j < 4; ++j)
                *reinterpret_cast<float4*>(tO + lane * 20 + 4 * j) = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
            __syncwarp();
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const float4 o4 = *reinterpret_cast<const float4*>(tO + (8 * i + r8) * 20 + 4 * p4);
                if (do_store && Rbase + 8 * i < a.Rows) *reinterpret_cast<float4*>(ybase + (long long)(8 * i) * a.y_cs + cg) = o4;
            }
            __syncwarp();
        }
    } else if (ups == 1) {
        float* yrow = a.y + (long long)b * a.y_bs + (long long)rc * a.y_cs;
        bool acc_r = a.accum != 0, mpost_r = a.mask_post != 0;
        if (a.split > 0) {          // WaveNet res/skip rows (wavenet.py:108-113)
            if (rc < a.split) { acc_r = true; mpost_r = true; }
            else { yrow = a.y2 + (long long)b * a.y2_bs + (long long)(rc - a.split) * a.y2_cs; acc_r = a.accum2 != 0; mpost_r = false; }
        }
        const float* rrow = a.res ? a.res + (long long)b * a.res_bs + (long long)rc * a.res_cs : nullptr;
        const float* mrow = a.ymask ? a.ymask + (long long)b * a.ymask_bs : nullptr;
        const int ycs_eff = (a.split > 0 && rc >= a.split) ? a.y2_cs : a.y_cs;
        const bool vec_ok = ((ycs_eff & 3) == 0) && (!a.res || (a.res_cs & 3) == 0) &&
                            ((reinterpret_cast<uintptr_t>(yrow) & 15) == 0) &&
                            (!rrow || (reinterpret_cast<uintptr_t>(rrow) & 15) == 0);
        // order-enforced software pipeline: the (volatile) loads of group j+1 are issued before the (volatile)
        // TMEM load of group j, into the OTHER of two register sets -- never copied (a move of a pending load's
        // result waits for the load and would serialise the groups).  float4 per lane along time (lane = one row).
        float rA[16], oA[16], rB[16], oB[16];
        auto prefetch = [&](int cg, float* r_, float* o_) {
            const int q = qb + cg;
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int qq = q + 4 * j;
                if (vec_ok && qq + 3 < a.Tout) {
                    if (rrow) asm volatile("ld.global.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(r_[4 * j]), "=f"(r_[4 * j + 1]), "=f"(r_[4 * j + 2]), "=f"(r_[4 * j + 3]) : "l"(rrow + qq));
                    if (acc_r) asm volatile("ld.global.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(o_[4 * j]), "=f"(o_[4 * j + 1]), "=f"(o_[4 * j + 2]), "=f"(o_[4 * j + 3]) : "l"(yrow + qq));
                } else {
#pragma unroll
                    for (int e = 0; e < 4; ++e) {
                        const int qe = min(qq + e, a.Tout - 1);
                        if (rrow) asm volatile("ld.global.f32 %0, [%1];" : "=f"(r_[4 * j + e]) : "l"(rrow + qe));
                        if (acc_r) asm volatile("ld.global.f32 %0, [%1];" : "=f"(o_[4 * j + e]) : "l"(yrow + qe));
                    }
                }
            }
        };
        const bool ld_ok = rok && !(a.dbg & 4), st_ok = rok && !(a.dbg & 8);
        auto group = [&](int cg, const float* rv, const float* ov, float* rn, float* on) {
            float v[16];
            if (ld_ok && cg + 16 < 128) prefetch(cg + 16, rn, on);
            tmem_ld16(dbase + (uint32_t)cg, v);
            const int q = qb + cg;
#pragma unroll
            for (int i = 0; i < 16; ++i) {
                float u = v[i] + bias;
                if (a.relu) u = fmaxf(u, 0.f);
                const float mk = mrow ? __ldg(mrow + min(q + i, a.Tout - 1)) : 1.f;
                if (a.mask_pre) u *= mk;
                if (a.res) u += rv[i];
                u *= a.scale;
                if (acc_r) u += ov[i];
                if (a.post_div != 1.f) u = u / a.post_div;
                if (mpost_r) u *= mk;
                v[i] = u;
            }
            if (st_ok) {
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const int qq = q + 4 * j;
                    if (vec_ok && qq + 3 < a.Tout) {
                        *reinterpret_cast<float4*>(yrow + qq) = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
                    } else {
#pragma unroll
                        for (int e = 0; e < 4; ++e) if (qq + e < a.Tout) yrow[qq + e] = v[4 * j + e];
                    }
                }
            }
        };
        if (ld_ok) prefetch(0, rA, oA);
#pragma unroll 1
        for (int cg = 0; cg < 128; cg += 32) {
            group(cg, rA, oA, rB, oB);
            group(cg + 16, rB, oB, rA, oA);
        }
    } else {
        // polyphase store: row r = co*ups + ph, column q -> y[co][q*ups + ph]; a warp's 32 lanes cover whole
        // groups of `ups` phases, i.e. contiguous runs of `ups` output samples per channel
        const int co = rc / ups, ph = rc - co * ups;
        float* yrow = a.y + (long long)b * a.y_bs + (long long)co * a.y_cs + ph;
        for (int cg = 0; cg < 128; cg += 16) {
            float v[16];
            tmem_ld16(dbase + (uint32_t)cg, v);
            if (!rok) continue;
#pragma unroll
            for (int i = 0; i < 16; ++i) {
                const int q = qb + cg + i;
                float u = v[i] + bias;
                if (a.relu) u = fmaxf(u, 0.f);
                const long long t = (long long)q * ups;
                if (q < a.Tq && t + ph < a.Tout) yrow[t] = u;
            }
        }
    }
}

// Out-of-line call of the general epilogue for the kernels whose hot path is the lean one (edge tiles only): inlined into
// their tile loop its loop invariants were hoisted across the lean path.  One copy of the arguments per call: through
// the reference every field use would be a generic load.
template <bool STAGED>
__device__ __noinline__ void general_tile_call(const Tc3Args& a_ref, unsigned char* smem, uint32_t tmem_base, uint32_t acc_cols,
                                               int b, int rt, int q0, int buf, int lq, int half, int lane, int warp) {
    const Tc3Args a = a_ref;
    general_tile_body<STAGED>(a, smem, tmem_base, acc_cols, b, rt, q0, buf, lq, half, lane, warp);
}

template <int GRP, bool STAGED = false, bool LEAN = true, bool X1 = false>   // GRP: tap groups stacked in the 128 MMA rows (1 = plain); STAGED: wide-layer
                                          // epilogue through per-warp shared tiles; LEAN: plain-layer kernel (lean epilogue inline, general
                                          // one out of line) -- false for the WaveNet / masked / transposed layers (general epilogue inline);
                                          // X1: single-pass TF32 (one rounded slab pair per operand, one MMA per tap)
__device__ __forceinline__ void tc3_body(const Tc3Args& a) {
    extern __shared__ __align__(128) unsigned char smem[];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int ROWS = a.rows_pad, RAWW = a.raw_w, K = a.KJ;
    const uint32_t rawStage = (uint32_t)KC2 * RAWS * 4;
    constexpr uint32_t NSL = X1 ? 2 : 4;                                 // slabs per stage / tap block
    const uint32_t slabA = (uint32_t)ROWS * 16, stageA = NSL * slabA;   // hi[2] + lo[2]  (single pass: x[2])
    const uint32_t slabB = (uint32_t)MROWS * 16, stageB = NSL * slabB;  // one tap block: {hi,lo}[2 slabs][128 rows][16 B]
    unsigned char* smRaw = smem;
    unsigned char* smA = smRaw + NRAW * rawStage;
    unsigned char* smB = smA + NA2 * stageA;
    uint64_t* bars = reinterpret_cast<uint64_t*>(smB + NB2 * stageB);
    const int A_FULL = 0, A_EMPTY = NA2, B_FULL = 2 * NA2, B_EMPTY = 2 * NA2 + NB2, ACC_FULL = 2 * NA2 + 2 * NB2,
              ACC_EMPTY = ACC_FULL + 2, NBARS = ACC_EMPTY + 2;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + NBARS);
    const uint32_t bar0 = smem_u32(bars);
    auto BAR = [&](int i) { return bar0 + 8u * (uint32_t)i; };

    const int nchunks = (a.Cin + KC2 - 1) / KC2;
    const bool ragged = a.lens != nullptr;
    int* pref = reinterpret_cast<int*>(smem + a.pref_off);    // pref[b] = first tile of row b (ragged only)
    if (ragged) {
        // tiles per row from its own length; exclusive prefix by warp 0 (rows in lane-contiguous chunks).  `lens` was
        // written several launches ago (durations kernel), so reading it before griddepcontrol.wait is safe.
        for (int b = tid; b < a.B; b += NTHREADS2) {
            const long long e = (long long)a.lens[b] * a.rate_q + a.need_q;
            const int ext = (int)(e < (long long)a.Tq ? (e > 0 ? e : 0) : (long long)a.Tq);
            pref[b + 1] = ((ext + a.tstep - 1) / a.tstep) * a.n_rtiles;
        }
        __syncthreads();
        if (warp == 0) {
            const int per = (a.B + 31) / 32, lo = lane * per, hi = min(a.B, lo + per);
            int sum = 0;
            for (int b = lo; b < hi; ++b) sum += pref[b + 1];
            int incl = sum;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) { const int n = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += n; }
            int run = incl - sum;
            for (int b = lo; b < hi; ++b) { const int c = pref[b + 1]; pref[b + 1] = run + c; run += c; }
            if (lane == 0) pref[0] = 0;
        }
        __syncthreads();
    }
    const int tiles_total = ragged ? pref[a.B] : a.B * a.n_rtiles * a.n_ttiles;
    const int my_tiles = (tiles_total > (int)blockIdx.x) ? (tiles_total - 1 - (int)blockIdx.x) / (int)gridDim.x + 1 : 0;
    const uint32_t acc_cols = (uint32_t)TT2;                     // per accumulator buffer
    const uint32_t ncols = 512;

    if (tid == 0) {
        for (int i = 0; i < NA2; ++i) { mbar_init(BAR(A_FULL + i), NPROD / 32); mbar_init(BAR(A_EMPTY + i), 1); }
        for (int i = 0; i < NB2; ++i) { mbar_init(BAR(B_FULL + i), 1); mbar_init(BAR(B_EMPTY + i), 1); }
        for (int i = 0; i < 2; ++i) { mbar_init(BAR(ACC_FULL + i), 1); mbar_init(BAR(ACC_EMPTY + i), 8); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == W_MMA) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(ncols) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    if constexpr (GRP == 1) {
        // Partial tiles issue MMAs over their valid columns only (MMA warp), so the epilogue can read accumulator columns
        // that no MMA of this launch wrote.  They are never consumed, but they may be stored past a row's extent and are
        // multiplied by the zero mask in the flow: make sure they are finite -- zero both accumulator buffers once.
        if (warp < 4 || warp >= W_EPI2) {
            const uint32_t zl = tmem_base + ((uint32_t)((warp & 3) * 32) << 16) + (uint32_t)((warp >= W_EPI2 ? 1 : 0) * 128);
#pragma unroll 1
            for (int c = 0; c < 128; c += 16) { tmem_st16_zero(zl + (uint32_t)c); tmem_st16_zero(zl + (uint32_t)(TT2 + c)); }
            tmem_wait_st();
        }
        tc_fence_before();
        __syncthreads();
        tc_fence_after();
    }
    if (tid == 0) TC3_STAMP(0);
    // Programmatic dependent launch: the next layer's CTAs may take SMs as this grid drains (they park in their own
    // griddepcontrol.wait); every role that touches activations waits for the previous layer here.  The weight loader
    // (warp W_LOAD) reads only constants and starts filling its ring at once.
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    if (warp != W_LOAD) asm volatile("griddepcontrol.wait;" ::: "memory");

    auto decode = [&](int it, int& b, int& rt, int& q0) {
        const int tile = (int)blockIdx.x + it * (int)gridDim.x;
        if (ragged) {
            int lo = 0, hi = a.B;                   // largest b with pref[b] <= tile (rows without tiles are skipped)
            while (hi - lo > 1) { const int mid = (lo + hi) >> 1; if (pref[mid] <= tile) lo = mid; else hi = mid; }
            b = lo;
            const int local = tile - pref[b], nt = (pref[b + 1] - pref[b]) / a.n_rtiles;
            rt = local / nt;
            q0 = (local - rt * nt) * a.tstep;
            return;
        }
        const int tt = tile % a.n_ttiles, rest = tile / a.n_ttiles;
        rt = rest % a.n_rtiles;
        b = rest / a.n_rtiles;
        q0 = tt * a.tstep;
    };
    auto input_extent = [&](int b) -> int {       // columns of x[b] that hold data; beyond it the operand is zero
        if (!ragged) return a.Tin;
        const long long e = (long long)a.lens[b] * a.rate_in + a.need_in;
        return (int)(e < (long long)a.Tin ? (e > 0 ? e : 0) : (long long)a.Tin);
    };

    if (warp >= W_PROD && warp < W_PROD + NPW) {
        // ============================================================ producers
        const int ptid = tid - 32 * W_PROD;
        const int total = my_tiles * nchunks;
        const int vec_per_row = RAWW / 4;
        const int nvec = KC2 * vec_per_row;
        const float slope = a.in_slope;
        const float* const xg = a.x;
        const long long x_bs = a.x_bs;
        const int x_cs = a.x_cs, Cin = a.Cin, pad = a.pad;
        const bool tracing = a.trace != nullptr;
        bool ok = true;
        // This loop paces every K <= 7 layer (r02 ncu source view: ~400 dependent instructions per warp and chunk, most of
        // them address arithmetic and bounds logic, ~2000 cycles).  So: per-thread work items are decoded ONCE (no
        // divisions in the loop), the raw row stride is a compile-time constant (shared loads take immediate offsets),
        // interior windows take a copy path without any bounds logic, and leaky ReLU is max(x, slope * x).
        constexpr int MAXV = (8 * 81 + NPROD - 1) / NPROD, MAXI = (2 * 320 + NPROD - 1) / NPROD;   // raw vectors / slab rows per thread
        int v_ch[MAXV], v_t[MAXV], v_src[MAXV];    // channel in chunk (-1: none), time offset from `tal`, global float offset
        uint32_t v_dst[MAXV];                      // byte offset in a raw stage
#pragma unroll
        for (int e = 0; e < MAXV; ++e) {
            const int v = ptid + e * NPROD;
            const int ch = v / vec_per_row, j = v - ch * vec_per_row;
            v_ch[e] = (v < nvec) ? ch : -1;
            v_t[e] = 4 * j;
            v_src[e] = ch * x_cs + 4 * j;
            v_dst[e] = (uint32_t)(ch * RAWS + 4 * j) * 4u;
        }
        int i_raw[MAXI], i_dst[MAXI];              // raw float offset of channel 0 of the slab row (-1: none), slab byte offset
#pragma unroll
        for (int e = 0; e < MAXI; ++e) {
            const int idx = ptid + e * NPROD;
            const int sl = idx / ROWS, r = idx - sl * ROWS;
            i_raw[e] = (idx < 2 * ROWS) ? (4 * sl) * RAWS + r : -1;
            i_dst[e] = (int)(sl * slabA) + r * 16;
        }
        // running positions instead of divisions / modulos per chunk
        int iss_it = 0, iss_c = 0, iss_ring = 0, iss_tal = 0, iss_Tin = 0;             // cp.async front: tile, chunk, raw slot
        const float* iss_row = xg;
        bool iss_new = true, iss_int = false;
        int tr_it = 0, tr_c = 0, tr_ring = 0, tr_q0 = 0, as = 0;                       // transform: tile, chunk, raw slot, A stage
        uint32_t pa_empty = 1;                                    // parity to wait for on A_EMPTY[as]: round 1 -> 0, round 2 -> 1, ...
        bool tr_new = true;
        const bool no_cp = (a.dbg & 1) != 0;
        const uint32_t raw_u32 = smem_u32(smRaw);
        auto issue = [&](int g) {
            if (g < total && !no_cp) {
                if (iss_new) {
                    int b_, rt_, q0_;
                    decode(iss_it, b_, rt_, q0_);
                    iss_Tin = input_extent(b_);
                    iss_tal = (q0_ - pad) & ~3;                            // 16-byte aligned window start (may be < 0)
                    iss_row = xg + (long long)b_ * x_bs;
                    iss_int = iss_tal >= 0 && iss_tal + RAWW <= iss_Tin && (Cin & (KC2 - 1)) == 0;
                    iss_new = false;
                }
                const uint32_t dst0 = raw_u32 + (uint32_t)iss_ring * rawStage;
                if (iss_int) {                                             // whole window inside the row: plain 16-byte copies
                    const float* src = iss_row + (long long)(iss_c * KC2) * x_cs + iss_tal;
#pragma unroll
                    for (int e = 0; e < MAXV; ++e)
                        if (v_ch[e] >= 0) cp_async16(dst0 + v_dst[e], src + v_src[e]);
                } else {
#pragma unroll
                    for (int e = 0; e < MAXV; ++e) {
                        if (v_ch[e] < 0) continue;
                        const int t = iss_tal + v_t[e];
                        const int cg = iss_c * KC2 + v_ch[e];
                        // t is a multiple of 4, so a vector is either wholly before the sequence start (zero fill),
                        // wholly inside, or cut by its end (partial source size, rest zero-filled by the hardware)
                        int nb = 0;
                        if (cg < Cin && t >= 0) nb = 4 * max(0, min(4, iss_Tin - t));
                        const int tsafe = (t >= 0 && t < iss_Tin) ? t : 0;
                        const float* src = iss_row + (long long)(cg < Cin ? cg : 0) * x_cs + tsafe;
                        cp_async16_zfill(dst0 + v_dst[e], src, (uint32_t)nb);
                    }
                }
                if (++iss_c == nchunks) { iss_c = 0; ++iss_it; iss_new = true; }
            }
            if (++iss_ring == NRAW) iss_ring = 0;
            asm volatile("cp.async.commit_group;" ::: "memory");
        };
        for (int g = 0; g < NRAW - 1; ++g) issue(g);
        for (int g = 0; g < total && ok; ++g) {
            asm volatile("cp.async.wait_group %0;" ::"n"(NRAW - 2) : "memory");
            named_bar_sync(1, NPROD);                                     // everyone's copies of chunk g have landed
            issue(g + NRAW - 1);                                          // refills the stage transformed last iteration
            if (g >= NA2) ok = mbar_wait(BAR(A_EMPTY + as), pa_empty, a.err);
            if (!ok) break;
            if (tr_new) {
                int b_, rt_;
                decode(tr_it, b_, rt_, tr_q0);
                tr_new = false;
            }
            const int tin0 = tr_q0 - pad, off = tin0 - (tin0 & ~3);
            const float* raw = reinterpret_cast<const float*>(smRaw + tr_ring * rawStage) + off;
            unsigned char* base = smA + as * stageA;
            if (!(a.dbg & 2)) {
                float u[MAXI][4];
#pragma unroll
                for (int e = 0; e < MAXI; ++e) {           // all shared loads first ...
                    const float* rp = raw + (i_raw[e] < 0 ? 0 : i_raw[e]);
#pragma unroll
                    for (int i = 0; i < 4; ++i) u[e][i] = rp[i * RAWS];
                }
#pragma unroll
                for (int e = 0; e < MAXI; ++e) {           // ... then prologue, hi/lo split and the two 16-byte stores
                    if (i_raw[e] < 0) continue;
                    if constexpr (X1) {                     // single pass: leaky ReLU, round to TF32, one store
                        float4 v;
                        float* pv = &v.x;
#pragma unroll
                        for (int i = 0; i < 4; ++i) pv[i] = tf32_rna(fmaxf(u[e][i], u[e][i] * slope));
                        *reinterpret_cast<float4*>(base + i_dst[e]) = v;
                        continue;
                    }
                    float4 hi, lo;
                    float* ph = &hi.x; float* pl = &lo.x;
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        const float w_ = fmaxf(u[e][i], u[e][i] * slope);        // leaky ReLU for 0 <= slope <= 1 (1: identity)
                        const float h = __uint_as_float(__float_as_uint(w_) & 0xFFFFE000u);
                        ph[i] = h;
                        pl[i] = w_ - h;
                    }
                    *reinterpret_cast<float4*>(base + i_dst[e]) = hi;
                    *reinterpret_cast<float4*>(base + 2 * slabA + i_dst[e]) = lo;
                }
            }
            fence_async_smem();
            __syncwarp();
            if (lane == 0) mbar_arrive(BAR(A_FULL + as));       // one arrival per producer warp
            if (++tr_c == nchunks) { tr_c = 0; ++tr_it; tr_new = true; }
            if (++tr_ring == NRAW) tr_ring = 0;
            if (++as == NA2) { as = 0; pa_empty ^= 1u; }
            if (tracing && ptid == 0) { if (g == 0) TC3_STAMP(1); if (g == nchunks - 1) TC3_STAMP(2); if (g == 2 * nchunks - 1) TC3_STAMP(3); if (g == 4 * nchunks - 1) TC3_STAMP(4); }
        }
        asm volatile("cp.async.wait_group 0;" ::: "memory");
        if (ptid == 0) TC3_STAMP(5);
    } else if (warp == W_LOAD) {
        // ============================================================ weight loader
        // One lane per ring slot: lane s owns slot s and feeds it with tap blocks s, s + NB2, s + 2*NB2, ... of this CTA's
        // block sequence.  A single thread walking the ring paid its wait -> expect_tx -> bulk-copy chain (~400 cycles) once
        // per 8 KB block -- measured as a 20 B/clk "L2 limit" that was really this thread (r02 ablation: the kernel without
        // MMAs still took 75 % of its time).  One independent chain per slot keeps NB2 copies in flight.
        if (lane < NB2) {
            const int total = nchunks * K;                                 // tap blocks per tile (contiguous in memory)
            const long long all = (long long)my_tiles * total;
            const uint32_t full = BAR(B_FULL + lane), empty = BAR(B_EMPTY + lane);
            const uint32_t dst = smem_u32(smB + lane * stageB);
            int it = 0, j = lane;                                          // block gi = it * total + j
            while (j >= total && it < my_tiles) { j -= total; ++it; }
            int cur_it = -1;
            const unsigned char* wsrc = nullptr;
            uint32_t par = 1;                                              // parity of B_EMPTY to wait for: round 1 -> 0, 2 -> 1
            bool ok = true, first = true;
            for (long long gi = lane; gi < all && ok; gi += NB2) {
                if (it != cur_it) {
                    int b_, rt, q0_;
                    decode(it, b_, rt, q0_);
                    wsrc = reinterpret_cast<const unsigned char*>(a.w) + (size_t)rt * total * stageB;
                    cur_it = it;
                }
                if (!first) { ok = mbar_wait(empty, par, a.err); if (!ok) break; }
                mbar_expect_tx(full, stageB);
                bulk_g2s(dst, wsrc + (size_t)j * stageB, stageB, full);
                first = false;
                par ^= 1u;
                j += NB2;
                while (j >= total) { j -= total; ++it; }
            }
        }
        __syncwarp();
    } else if (warp == W_MMA) {
        // ============================================================ MMA issuer
        // ncu (profiles/r02_tc3_issue_loop.md): this ONE thread is what bounds the MMA-heavy layers -- it never waits long
        // on a barrier, its own dependent instruction chain took ~710 cycles per tap against the 384 cycles the three MMAs
        // need on the tensor pipe.  So the loop carries no divisions / modulos / constant-bank loads / descriptor
        // rebuilds: ring positions, parities, barrier addresses and descriptors are running counters, and the next tap's
        // weight barrier is tested (non-blocking) BEFORE the current tap's MMAs are issued so its latency is off the chain.
        // The whole warp runs the loop CONVERGED (every lane computes the same ring positions / descriptors, so the
        // compiler keeps them in uniform registers and feeds UTCHMMA directly -- inside an `if (lane == 0)` every operand
        // went through R2UR and each tcgen05 instruction got its own ELECT loop); one elected lane issues.
        {
            uint32_t leader;
            asm volatile("{\n.reg .pred p;\nelect.sync _|p, 0xffffffff;\nselp.u32 %0, 1, 0, p;\n}" : "=r"(leader));
            // M = 128 rows (weights), N = 256 time steps
            const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(TT2 >> 3) << 17) | ((uint32_t)(MROWS >> 4) << 24);
            const uint64_t xstep = (uint64_t)a.dil_blk;                                   // B rows per tap (16 B each)
            const uint64_t wlo_off = (uint64_t)((2 * slabB) >> 4), wslot = (uint64_t)(stageB >> 4);
            const uint64_t wdesc0 = make_desc(smem_u32(smB), slabB);
            const uint32_t bfull0 = BAR(B_FULL), bempty0 = BAR(B_EMPTY);
            const bool no_mma = (a.dbg & 16) != 0;
#ifdef TC3_RACE_PROBE      // harness-only sanitizer probe (tools/r2u.sh): plain mbarrier arrivals instead of tcgen05.commit
            const bool thread_arrive = no_mma && (a.dbg & 256) != 0;
#else
            constexpr bool thread_arrive = false;
#endif
            const bool no_probe = (a.dbg & 64) != 0;                                       // every weight barrier through try_wait
            bool ok = true;
            int sa = 0; uint32_t pa = 0;                                                  // activation stage / its parity
            int sb = 0; uint32_t pb = 0;                                                  // weight slot / its parity
            uint64_t wdesc = wdesc0;
            uint32_t bfull = bfull0, bempty = bempty0;
            bool have = false;                                                            // B_FULL[sb] already seen complete
            for (int it = 0; it < my_tiles && ok; ++it) {
                const int buf = it & 1;
                if (it >= 2) ok = mbar_wait(BAR(ACC_EMPTY + buf), ((it >> 1) - 1) & 1, a.err);
                if (!ok) break;
                tc_fence_after();
                const uint32_t dcol = tmem_base + (uint32_t)buf * acc_cols;
                uint32_t acc = 0u;
                // The last tile of a row is on average half empty (the single tile of a flow / conv_pre row even more): its
                // MMAs cover only the columns that hold data, N = 16 * ceil(valid / 16).  Columns beyond stay stale in TMEM;
                // the epilogue may store them past the row's extent, where no consumer reads (consumer extents <= producer
                // extents by construction of the margins) and the final waveform tail is zero-filled by conv_post.
                uint32_t idesc_t = idesc;
                if constexpr (GRP == 1) {
                    if (!(a.dbg & 512)) {
                        int b_, rt_, q0_;
                        decode(it, b_, rt_, q0_);
                        long long ext = a.Tq;
                        if (ragged) {
                            const long long e = (long long)a.lens[b_] * a.rate_q + a.need_q;
                            ext = e < (long long)a.Tq ? (e > 0 ? e : 0) : (long long)a.Tq;
                        }
                        int n = ((int)ext - q0_ + 15) & ~15;
                        n = n < 16 ? 16 : (n > TT2 ? TT2 : n);
                        idesc_t = (idesc & ~(0x3Fu << 17)) | ((uint32_t)(n >> 3) << 17);
                    }
                }
                for (int c = 0; c < nchunks && ok; ++c) {
                    ok = mbar_wait(BAR(A_FULL + sa), pa, a.err);
                    if (!ok) break;
                    tc_fence_after();
                    const uint32_t abase = smem_u32(smA + sa * stageA);
                    // descriptors differ only in the 14-bit start-address field: build once, then add rows (16 B each)
                    uint64_t xh = make_desc(abase, slabA), xl = make_desc(abase + 2 * slabA, slabA);
#pragma unroll 1
                    for (int k = 0; k < K; ++k) {
                        if (!have) { ok = mbar_wait(bfull, pb, a.err); if (!ok) break; }
                        tc_fence_after();
                        // where the NEXT tap's weights will be; peek at their barrier now (result used next iteration)
                        const bool wrap = (sb == NB2 - 1);
                        const uint32_t nfull = wrap ? bfull0 : bfull + 8u, npb = wrap ? (pb ^ 1u) : pb;
                        const bool have_next = no_probe ? false : mbar_test(nfull, npb);
                        const uint64_t w_hi = wdesc, w_lo = wdesc + wlo_off;
                        if (leader) {
                            if (!no_mma) {
                                if constexpr (X1) {
                                    mma_tf32(dcol, w_hi, xh, idesc_t, acc);
                                } else {
                                    mma_tf32(dcol, w_hi, xl, idesc_t, acc);               // small terms first
                                    mma_tf32(dcol, w_lo, xh, idesc_t, 1u);
                                    mma_tf32(dcol, w_hi, xh, idesc_t, 1u);
                                }
                            }
                            if (thread_arrive) mbar_arrive(bempty); else mma_commit(bempty);
                        }
                        acc = 1u;
                        xh += xstep; xl += xstep;
                        if (wrap) { sb = 0; wdesc = wdesc0; bempty = bempty0; }
                        else { ++sb; wdesc += wslot; bempty += 8u; }
                        bfull = nfull; pb = npb;
                        have = __all_sync(0xffffffffu, have_next);                        // keep the warp's control flow uniform
                    }
                    if (ok && leader) { if (thread_arrive) mbar_arrive(BAR(A_EMPTY + sa)); else mma_commit(BAR(A_EMPTY + sa)); }
                    if (++sa == NA2) { sa = 0; pa ^= 1u; }
                }
                if (ok && leader) { if (thread_arrive) mbar_arrive(BAR(ACC_FULL + buf)); else mma_commit(BAR(ACC_FULL + buf)); }
                if (lane == 0) { if (it == 0) TC3_STAMP(8); if (it == 1) TC3_STAMP(9); if (it == 3) TC3_STAMP(10); }
            }
            if (lane == 0) TC3_STAMP(11);
        }
        __syncwarp();
    } else {
        // ============================================================ epilogue (lane = output row, columns = time)
        bool ok = true;
        const int ups = a.ups;
        const int lq = warp & 3;                     // TMEM lane quarter this warp may access
        const int half = (warp >= W_EPI2) ? 1 : 0;   // warps 0-3: columns [0,128), warps W_EPI2..+3: [128,256)
        if constexpr (GRP > 1) {
            // ---- grouped epilogue: out[c, t] = sum_g D_g[c, t + g*dil].  MMA row m = g * CH + c (CH = 128 / GRP channels), so a
            // warp's TMEM lane quarter holds ONE tap group (GRP = 4) or half of one (GRP = 2) and applies that group's shift as
            // a plain column offset of its tcgen05.ld -- no per-lane selects.  The GRP partials of a channel live in different
            // warps; the four warps of a column half exchange them through a double-buffered shared tile (one named barrier
            // per 16-column group), after which thread (c, j) owns float4 j of channel c: 4 lanes = 64 contiguous bytes.
            // r02 measurement behind this (profiles/r02_epilogue_instruction_bound.md): the previous shuffle reduce-scatter
            // cost ~180 instructions per lane and 16 columns and paced the narrow layers (3.3 us per tile with no memory ops).
            constexpr int CH = 128 / GRP;              // output channels
            constexpr int NQ = CH / 32;                // float4 per thread and 16-column group (1 or 2)
            constexpr int NV = 4 * NQ;
            const int tq = lq * 32 + lane;             // thread within the half's four warps == its TMEM row
            const int gq = (lq * 32) / CH;             // tap group of this warp's TMEM lanes
            const int cw = tq - gq * CH;               // channel of this lane's TMEM row
            const int co = (tq * NQ) >> 2;             // channel this thread finishes
            const int j0 = (tq & (4 / NQ - 1)) * NQ;   // its first float4 within a 16-column group
            const int coff = 4 * j0;
            const int cbeg = half ? 128 : 0;
            const bool has_res = a.res != nullptr && !(a.dbg & 4);
            const bool acc_r = a.accum != 0 && !(a.dbg & 4);
            const bool vec_ok = ((a.y_cs & 3) == 0) && ((a.y_bs & 3) == 0) && ((reinterpret_cast<uintptr_t>(a.y) & 15) == 0) &&
                                (!a.res || (((a.res_cs & 3) == 0) && ((a.res_bs & 3) == 0) && ((reinterpret_cast<uintptr_t>(a.res) & 15) == 0)));
            const bool relu = a.relu != 0, do_store = !(a.dbg & 8);
            const float scale = a.scale, post_div = a.post_div;
            const bool plain = !relu && scale == 1.f;
            float* xq = reinterpret_cast<float*>(smem + a.stage_off) + half * 4096;        // two buffers of [128 rows][16] floats
            const int wsw = (cw >> 1) & 3, rsw = (co >> 1) & 3;                             // 16-byte unit swizzle (bank spread)
            float* xw = xq + tq * 16;
            const uint32_t gshift = (uint32_t)(gq * a.dil);
            const int bar_id = 2 + half;
            int xbuf = 0;
            bool fast = false;                                            // interior tile: no bounds checks at all
            auto prefetch_any = [&](const float* rr, int q, float* dst) {   // values of one column group of a row -> registers
#pragma unroll
                for (int j = 0; j < NQ; ++j) {
                    const int qq = q + 4 * j;
                    if (fast || (vec_ok && qq + 3 < a.Tout)) {
                        asm volatile("ld.global.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(dst[4 * j]), "=f"(dst[4 * j + 1]), "=f"(dst[4 * j + 2]), "=f"(dst[4 * j + 3]) : "l"(rr + qq));
                    } else {
#pragma unroll
                        for (int e = 0; e < 4; ++e) asm volatile("ld.global.f32 %0, [%1];" : "=f"(dst[4 * j + e]) : "l"(rr + min(qq + e, a.Tout - 1)));
                    }
                }
            };
            auto prefetch = [&](const float* rr, int q, float* dst) { if (has_res) prefetch_any(rr, q, dst); };
            auto prefetch_acc = [&](const float* rr, int q, float* dst) { if (rr) prefetch_any(rr, q, dst); };
            for (int it = 0; it < my_tiles && ok; ++it) {
                const int buf = it & 1;
                int b, rt, q0;
                decode(it, b, rt, q0);
                const float* rrow = has_res ? a.res + (long long)b * a.res_bs + (long long)co * a.res_cs : nullptr;
                const int cend = half ? a.tstep : min(128, a.tstep);
                fast = vec_ok && (q0 + a.tstep <= a.Tout);
                // Residual / accumulate values are prefetched TWO column groups ahead into three rotating register sets that
                // are never copied (a register move of a pending load's result waits for the load).
                float rA[NV], rB[NV], rC[NV], oA[NV], oB[NV], oC[NV];
                float* yrow = a.y + (long long)b * a.y_bs + (long long)co * a.y_cs;
                const float* orow = acc_r ? yrow : nullptr;
                // the first two column groups are requested before waiting for the accumulator
                prefetch(rrow, q0 + cbeg + coff, rA);
                prefetch_acc(orow, q0 + cbeg + coff, oA);
                if (cbeg + 16 < cend) { prefetch(rrow, q0 + cbeg + 16 + coff, rB); prefetch_acc(orow, q0 + cbeg + 16 + coff, oB); }
                ok = mbar_wait(BAR(ACC_FULL + buf), (it >> 1) & 1, a.err);
                if (!ok) break;
                tc_fence_after();
                if (tid == 0) { if (it == 0) TC3_STAMP(16); if (it == 1) TC3_STAMP(18); if (it == 3) TC3_STAMP(20); }
                if (a.dbg & 32) { tc_fence_before(); __syncwarp(); if (lane == 0) mbar_arrive(BAR(ACC_EMPTY + buf)); continue; }   // probe: handshake only
                const uint32_t dlane = tmem_base + (uint32_t)buf * acc_cols + ((uint32_t)(lq * 32) << 16) + gshift;
                float bias = a.bias[co];
                if (a.cond) bias += __ldg(a.cond + (long long)b * a.cond_bs + co);
                uint32_t P[16];
                tmem_ld16_nowait(dlane + (uint32_t)cbeg, P);                 // this warp's partial of the first column group
                auto group = [&](int cg, const float* rv, const float* ov, float* rf, float* of) {
                    if (cg + 32 < cend) { prefetch(rrow, q0 + cg + 32 + coff, rf); prefetch_acc(orow, q0 + cg + 32 + coff, of); }
                    float* xb = xw + xbuf * 2048;
                    tmem_wait_ld();
#pragma unroll
                    for (int j = 0; j < 4; ++j)
                        *reinterpret_cast<uint4*>(xb + 4 * (j ^ wsw)) = make_uint4(P[4 * j], P[4 * j + 1], P[4 * j + 2], P[4 * j + 3]);
                    if (cg + 16 < cend) tmem_ld16_nowait(dlane + (uint32_t)(cg + 16), P);   // next group's partial flies during the exchange
                    else {                                                                   // last TMEM read of this tile: release the accumulator
                        tc_fence_before();
                        __syncwarp();
                        if (lane == 0) mbar_arrive(BAR(ACC_EMPTY + buf));
                    }
                    named_bar_sync(bar_id, 128);
                    const float* xr = xq + xbuf * 2048 + co * 16;
                    xbuf ^= 1;
                    float R[NV];
#pragma unroll
                    for (int e = 0; e < NQ; ++e) {
                        const int u4 = 4 * ((j0 + e) ^ rsw);
                        const float4 p0 = *reinterpret_cast<const float4*>(xr + u4);
                        const float4 p1 = *reinterpret_cast<const float4*>(xr + CH * 16 + u4);
                        float4 s = make_float4(p0.x + p1.x, p0.y + p1.y, p0.z + p1.z, p0.w + p1.w);
                        if constexpr (GRP == 4) {
                            const float4 p2 = *reinterpret_cast<const float4*>(xr + 2 * CH * 16 + u4);
                            const float4 p3 = *reinterpret_cast<const float4*>(xr + 3 * CH * 16 + u4);
                            const float4 s2 = make_float4(p2.x + p3.x, p2.y + p3.y, p2.z + p3.z, p2.w + p3.w);
                            s = make_float4(s.x + s2.x, s.y + s2.y, s.z + s2.z, s.w + s2.w);
                        }
                        R[4 * e] = s.x; R[4 * e + 1] = s.y; R[4 * e + 2] = s.z; R[4 * e + 3] = s.w;
                    }
                    if (plain) {
#pragma unroll
                        for (int i = 0; i < NV; ++i) {
                            float u = R[i] + bias;
                            if (has_res) u += rv[i];
                            if (acc_r) u += ov[i];
                            R[i] = u;
                        }
                        if (post_div != 1.f) {
#pragma unroll
                            for (int i = 0; i < NV; ++i) R[i] = R[i] / post_div;
                        }
                    } else {
#pragma unroll
                        for (int i = 0; i < NV; ++i) {
                            float u = R[i] + bias;
                            if (relu) u = fmaxf(u, 0.f);
                            if (has_res) u += rv[i];
                            u *= scale;
                            if (acc_r) u += ov[i];
                            if (post_div != 1.f) u = u / post_div;
                            R[i] = u;
                        }
                    }
                    if (do_store) {
                        const int q = q0 + cg + coff;
#pragma unroll
                        for (int j = 0; j < NQ; ++j) {
                            const int qq = q + 4 * j;
                            if (fast || (vec_ok && qq + 3 < a.Tout)) {
                                *reinterpret_cast<float4*>(yrow + qq) = make_float4(R[4 * j], R[4 * j + 1], R[4 * j + 2], R[4 * j + 3]);
                            } else {
#pragma unroll
                                for (int e = 0; e < 4; ++e) if (qq + e < a.Tout) yrow[qq + e] = R[4 * j + e];
                            }
                        }
                    }
                };
#pragma unroll 1
                for (int cg = cbeg; cg < cend; cg += 48) {
                    group(cg, rA, oA, rC, oC);
                    if (cg + 16 < cend) group(cg + 16, rB, oB, rA, oA);
                    if (cg + 32 < cend) group(cg + 32, rC, oC, rB, oB);
                }
                if (tid == 0) { if (it == 0) TC3_STAMP(17); if (it == 1) TC3_STAMP(19); if (it == 3) TC3_STAMP(21); }
            }
            if (tid == 0) TC3_STAMP(22);
        } else {
        // launch-uniform part of the lean-path test (the per-tile part: the tile half lies wholly inside the row)
        const bool lean_launch = LEAN && ups == 1 && !a.gate && a.split == 0 && !a.relu && !a.ymask && a.scale == 1.f && a.post_div == 1.f &&
                                 !(STAGED && a.stage) &&
                                 ((a.y_cs & 3) == 0) && ((a.y_bs & 3) == 0) && ((reinterpret_cast<uintptr_t>(a.y) & 15) == 0) &&
                                 (!a.res || (((a.res_cs & 3) == 0) && ((a.res_bs & 3) == 0) && ((reinterpret_cast<uintptr_t>(a.res) & 15) == 0)));
        const bool hres = a.res != nullptr && !(a.dbg & 4), hacc = a.accum != 0 && !(a.dbg & 4), do_st = !(a.dbg & 8);
        float* const lean_tiles = (!STAGED && a.stage_off > 0 && !(a.dbg & 128)) ? reinterpret_cast<float*>(smem + a.stage_off) : nullptr;
        for (int it = 0; it < my_tiles && ok; ++it) {
            const int buf = it & 1;
            int b, rt, q0;
            decode(it, b, rt, q0);
            ok = mbar_wait(BAR(ACC_FULL + buf), (it >> 1) & 1, a.err);
            if (!ok) break;
            tc_fence_after();
            if (tid == 0) { if (it == 0) TC3_STAMP(16); if (it == 1) TC3_STAMP(18); if (it == 3) TC3_STAMP(20); }
            if (a.dbg & 32) { tc_fence_before(); __syncwarp(); if (lane == 0) mbar_arrive(BAR(ACC_EMPTY + buf)); continue; }   // probe: handshake only
            const int qb = q0 + half * 128;
            if (LEAN && lean_launch && qb + 128 <= a.Tout) {
                // ---- lean path: every interior tile of the plain layers (bias, optional residual / accumulate).  r02 ncu
                // source view of the general loop: ~1000 instructions per lane and 16 columns on options that are off, the
                // eight epilogue warps issue bound.
                const int r = rt * MROWS + lq * 32 + lane;             // GEMM row of this lane
                const bool rok = r < a.Rows;
                const int rc = rok ? r : a.Rows - 1;
                const uint32_t dbase = tmem_base + (uint32_t)buf * acc_cols + ((uint32_t)(lq * 32) << 16) + (uint32_t)(half * 128);
                float bias = a.bias[rc];
                if (a.cond) bias += __ldg(a.cond + (long long)b * a.cond_bs + rc);
                const bool st_ok = do_st && rok;
                float* yp = a.y + (long long)b * a.y_bs + (long long)rc * a.y_cs + qb;
                const float* rp = hres ? a.res + (long long)b * a.res_bs + (long long)rc * a.res_cs + qb : yp;
                if (lean_tiles) {                                  // transposing variant: coalesced global accesses
                    float* tO = lean_tiles + ((warp < 4) ? warp : warp - W_EPI2 + 4) * LEAN_TILE_FLOATS;
                    float* yq = a.y + (long long)b * a.y_bs + qb;
                    const float* rq = hres ? a.res + (long long)b * a.res_bs + qb : yq;
                    const int row0 = rt * MROWS + lq * 32;
                    if (hres) { if (hacc) lean_rows_t<true, true>(dbase, bias, tO, lane, rq, yq, a.res_cs, a.y_cs, row0, a.Rows, do_st);
                                else lean_rows_t<true, false>(dbase, bias, tO, lane, rq, yq, a.res_cs, a.y_cs, row0, a.Rows, do_st); }
                    else { if (hacc) lean_rows_t<false, true>(dbase, bias, tO, lane, rq, yq, 0, a.y_cs, row0, a.Rows, do_st);
                           else lean_rows_t<false, false>(dbase, bias, tO, lane, rq, yq, 0, a.y_cs, row0, a.Rows, do_st); }
                } else if (hres) { if (hacc) lean_rows<true, true>(dbase, bias, rp, yp, st_ok); else lean_rows<true, false>(dbase, bias, rp, yp, st_ok); }
                else { if (hacc) lean_rows<false, true>(dbase, bias, rp, yp, st_ok); else lean_rows<false, false>(dbase, bias, rp, yp, st_ok); }
            } else {
                if constexpr (LEAN) general_tile_call<STAGED>(a, smem, tmem_base, acc_cols, b, rt, q0, buf, lq, half, lane, warp);
                else general_tile_body<STAGED>(a, smem, tmem_base, acc_cols, b, rt, q0, buf, lq, half, lane, warp);
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(BAR(ACC_EMPTY + buf));   // one arrival per epilogue warp
            if (tid == 0) { if (it == 0) TC3_STAMP(17); if (it == 1) TC3_STAMP(19); if (it == 3) TC3_STAMP(21); }
        }
        if (tid == 0) TC3_STAMP(22);
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == W_MMA) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(ncols) : "memory");
    }
}

__global__ void __launch_bounds__(NTHREADS2, 1) conv1d_tc3_kernel(const __grid_constant__ Tc3Args a) { tc3_body<1>(a); }
__global__ void __launch_bounds__(NTHREADS2, 1) conv1d_tc3s_kernel(const __grid_constant__ Tc3Args a) { tc3_body<1, true, false>(a); }
__global__ void __launch_bounds__(NTHREADS2, 1) conv1d_tc3x_kernel(const __grid_constant__ Tc3Args a) { tc3_body<1, false, false>(a); }   // gate / split / mask / polyphase
template <int GRP>
__global__ void __launch_bounds__(NTHREADS2, 1) conv1d_tc3g_kernel(const __grid_constant__ Tc3Args a) { tc3_body<GRP>(a); }
// single-pass TF32 twins (no staged one: a single-pass layer never takes the staged epilogue)
__global__ void __launch_bounds__(NTHREADS2, 1) conv1d_tc3_tf32_kernel(const __grid_constant__ Tc3Args a) { tc3_body<1, false, true, true>(a); }
__global__ void __launch_bounds__(NTHREADS2, 1) conv1d_tc3x_tf32_kernel(const __grid_constant__ Tc3Args a) { tc3_body<1, false, false, true>(a); }
template <int GRP>
__global__ void __launch_bounds__(NTHREADS2, 1) conv1d_tc3g_tf32_kernel(const __grid_constant__ Tc3Args a) { tc3_body<GRP, false, true, true>(a); }

typedef void (*Tc3Kernel)(const Tc3Args);
// grouped kernel for 2 / 4 tap groups (any dilation with (GRP - 1) * dil <= 15); x1: single-pass TF32
static inline Tc3Kernel grouped_kernel(int grp, bool x1 = false) {
    if (x1) return grp == 2 ? conv1d_tc3g_tf32_kernel<2> : conv1d_tc3g_tf32_kernel<4>;
    return grp == 2 ? conv1d_tc3g_kernel<2> : conv1d_tc3g_kernel<4>;
}
constexpr int GROUP_XCHG_BYTES = 2 * 2 * 128 * 16 * 4;   // grouped epilogue: per column half two buffers of [128 rows][16] floats

}  // namespace tc3
}  // namespace b200tts
