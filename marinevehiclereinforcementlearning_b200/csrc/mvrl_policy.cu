// Fused actor for rollout collection (BASELINE.json config 5; SURVEY.md 8(f) N2 / 8(d) cfg 5): the policy network of
// tag_00_Dec2023_simpleControlTurbulence/main_00_sbl.py:100-105 (MlpPolicy, net_arch [128, 128, 128], GELU) plus the
// Gaussian action head, as ONE kernel that reads the env's structure-of-arrays observation buffer in place and writes the
// structure-of-arrays action buffer the step kernel reads: obs [O][ld] -> 128 -> 128 -> 128 -> A, tanh mean, a = clip(mean +
// std * eps, -1, 1), log-prob.  A rollout step is then two launches (this kernel + the fused env step).
//
// This is the dense contraction next to the path, so it runs on the tensor cores.  Two implementations live in this file:
//
//  * policy_act_tc5_kernel (namespace tc5, the default): written for the 5th-generation tensor core - tcgen05.mma with M = 128
//    (one tile = 128 environments = the 128 lanes of tensor memory), operands through shared-memory matrix descriptors,
//    fp32 accumulators in TMEM, the epilogue of a layer writing the next layer's A operand.  Description above the kernel.
//  * policy_act_kernel (MVRL_POLICY_MMA_SYNC=1): warp-level mma.sync m16n8k16; each warp owns 16 environments and the
//    16 x 128 activations never leave its registers - the accumulator fragment of one layer IS the A-operand fragment of
//    the next after bias + GELU + bf16 packing.  The weights (70 KB as bf16, pre-packed on the host in B-fragment order) sit
//    in shared memory; persistent grid, 2 CTAs per SM.  It re-reads every weight fragment for each 16 rows (587 MB of
//    shared-memory traffic per 131 072-env launch) and takes 42 us where the tcgen05 kernel takes 23; it stays as the
//    second implementation the tests compare the default against (same bf16 rounding, GELU code and Philox streams).
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <new>
#include <vector>

#include "mvrl_host.h"
#include "mvrl_math.cuh"

using namespace mvrl;

#ifndef MVRL_POLICY_PREFETCH
#define MVRL_POLICY_PREFETCH 1
#endif

namespace {

constexpr int H = 128;            // hidden width
constexpr int KIN = 16;           // observation dim padded to one k-step
constexpr int NOUT = 8;           // action dim padded to one n-tile
constexpr int TILE = 128;         // environments per CTA tile (8 warps x 16)
constexpr int THREADS = 256;

// byte offsets inside the packed parameter block (device + shared memory)
constexpr int OFF_W1 = 0;                          // [1 kk][16 nt][32 lanes] uint2
constexpr int OFF_W2 = OFF_W1 + 1 * 16 * 256;      // [8][16][32] uint2
constexpr int OFF_W3 = OFF_W2 + 8 * 16 * 256;
constexpr int OFF_W4 = OFF_W3 + 8 * 16 * 256;      // [8][1][32] uint2
constexpr int OFF_B = OFF_W4 + 8 * 1 * 256;        // float b1[128] b2[128] b3[128] b4[8] std[8]
constexpr int PACKED_BYTES = OFF_B + (3 * H + 2 * NOUT) * 4;
static_assert(PACKED_BYTES % 16 == 0, "packed block is copied with 16-byte accesses");
// squashed head (SB3 SAC / TQC Actor): b4[8] holds b_mu and std[8] holds b_log_std; the B fragments of the log_std layer
// follow the block, so that the fixed head's layout (and its kernel) stays as it is
constexpr int OFF_WLS = PACKED_BYTES;              // [8][1][32] uint2
constexpr int PACKED_BYTES_SQUASHED = OFF_WLS + 8 * 1 * 256;

constexpr int HEAD_FIXED = MVRL_POLICY_HEAD_FIXED_STD;
constexpr int HEAD_SQUASHED = MVRL_POLICY_HEAD_SQUASHED;
constexpr int packed_bytes(int head) { return head == HEAD_SQUASHED ? PACKED_BYTES_SQUASHED : PACKED_BYTES; }

struct PolicyArgs {
    const unsigned char* packed;
    long n, ld;
    const float* obs; float* act; float* logp; float* mean; float* eps;
    int obs_dim, act_dim, deterministic;
    float logp_const;
    unsigned long long seed, env_id0;
    unsigned step;
    // squashed head only (appended: the fixed-head kernels read the members above at unchanged offsets)
    float* log_std;              // nullable [act_dim][ld]: the clamped log std
    int noise;                   // 1: act = clip(a + noise_std * xi, -1, 1), xi ~ N(0, 1) from Philox stream 8
    float noise_std[NOUT];
};

__device__ __forceinline__ void mma_bf16(float (&c)[4], const unsigned (&a)[4], uint2 b) {
    asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                 : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
                 : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b.x), "r"(b.y));
}
__device__ __forceinline__ unsigned pack_bf16(float lo, float hi) {
    const __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);   // .x (low half) = lo
    return *reinterpret_cast<const unsigned*>(&v);
}
__device__ __forceinline__ float tanh_fast(float x) {
    float y;
    asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
// GELU in its tanh form, 0.5 x (1 + tanh(sqrt(2/pi) (x + 0.044715 x^3))) = torch gelu(approximate="tanh") - within 1e-3 of
// the erf form that torch.nn.GELU() (the reference's activation_fn, legacy/main_00_sbl.py:100-105) evaluates, i.e. below the
// bf16 operand rounding of this kernel
// bias + GELU of two adjacent columns at once on the packed fp32 instructions of sm_100 (FADD2 / FMUL2 / FFMA2: the
// activation is ~55 % of this kernel's instructions when written per element), then one bf16x2 pack
__device__ __forceinline__ unsigned gelu_pack2(float x0, float x1, float2 b) {
    const float2 x = __fadd2_rn(make_float2(x0, x1), b);
    const float2 x2 = __fmul2_rn(x, x);
    const float2 u = __fmul2_rn(x, __ffma2_rn(x2, make_float2(0.0356774081f, 0.0356774081f), make_float2(0.7978845608f, 0.7978845608f)));
    const float2 th = make_float2(tanh_fast(u.x), tanh_fast(u.y));
    const float2 h = __fmul2_rn(x, make_float2(0.5f, 0.5f));
    const float2 y = __ffma2_rn(h, th, h);
    return pack_bf16(y.x, y.y);
}

// 2 gelu(x) = x (1 + tanh(u)) of two columns, bias already in the accumulator: the tcgen05 kernel stores TWICE the activation
// and the host halves the next layer's weights (a power of two: exact in bf16 and in the fp32 accumulation, so nothing changes
// numerically) - one packed multiply fewer per pair of columns
__device__ __forceinline__ unsigned gelu2x_pack2(float x0, float x1) {
    const float2 x = make_float2(x0, x1);
    const float2 x2 = __fmul2_rn(x, x);
    const float2 u = __fmul2_rn(x, __ffma2_rn(x2, make_float2(0.0356774081f, 0.0356774081f), make_float2(0.7978845608f, 0.7978845608f)));
    const float2 th = make_float2(tanh_fast(u.x), tanh_fast(u.y));
    const float2 y = __ffma2_rn(x, th, x);
    return pack_bf16(y.x, y.y);
}
__device__ __forceinline__ unsigned gelu_pack2(float x0, float x1) {   // the same without the bias (already in the accumulator)
    const float2 x = make_float2(x0, x1);
    const float2 x2 = __fmul2_rn(x, x);
    const float2 u = __fmul2_rn(x, __ffma2_rn(x2, make_float2(0.0356774081f, 0.0356774081f), make_float2(0.7978845608f, 0.7978845608f)));
    const float2 th = make_float2(tanh_fast(u.x), tanh_fast(u.y));
    const float2 h = __fmul2_rn(x, make_float2(0.5f, 0.5f));
    const float2 y = __ffma2_rn(h, th, h);
    return pack_bf16(y.x, y.y);
}

// accumulators of one layer (+ bias, GELU) -> A fragments of the next: n-tiles 2kk and 2kk + 1 give k-step kk
__device__ __forceinline__ void activate_to_frags(const float (&acc)[16][4], const float* bias, int t, unsigned (&afr)[8][4]) {
#pragma unroll
    for (int kk = 0; kk < 8; ++kk) {
        const float2 b0 = *reinterpret_cast<const float2*>(bias + 16 * kk + 2 * t);
        const float2 b1 = *reinterpret_cast<const float2*>(bias + 16 * kk + 8 + 2 * t);
        const float (&c0)[4] = acc[2 * kk];
        const float (&c1)[4] = acc[2 * kk + 1];
        afr[kk][0] = gelu_pack2(c0[0], c0[1], b0);   // row g,     k = 16 kk + 2t, +1
        afr[kk][1] = gelu_pack2(c0[2], c0[3], b0);   // row g + 8
        afr[kk][2] = gelu_pack2(c1[0], c1[1], b1);   // row g,     k = 16 kk + 8 + 2t, +1
        afr[kk][3] = gelu_pack2(c1[2], c1[3], b1);   // row g + 8
    }
}

__device__ __forceinline__ void hidden_layer(const uint2* w, const unsigned (&afr)[8][4], int lane, float (&acc)[16][4]) {
#pragma unroll
    for (int nt = 0; nt < 16; ++nt) { acc[nt][0] = acc[nt][1] = acc[nt][2] = acc[nt][3] = 0.0f; }
#pragma unroll
    for (int kk = 0; kk < 8; ++kk) {
#pragma unroll
        for (int nt = 0; nt < 16; ++nt) mma_bf16(acc[nt], afr[kk], w[(kk * 16 + nt) * 32 + lane]);
    }
}

// two standard normals from one Philox block of (seed, environment, step): Box-Muller on 24-bit uniforms.  Stream 7 is the
// policy's eps, stream 8 the squashed head's action noise
constexpr unsigned STREAM_EPS = 7u, STREAM_NOISE = 8u;
__device__ __forceinline__ float2 normal_pair(unsigned long long seed, unsigned long long env, unsigned step, unsigned blk,
                                              unsigned stream = STREAM_EPS) {
    const uint4 w = Philox::draw(seed, env, step, stream, blk);
    const float u1 = (float(w.x >> 8) + 0.5f) * (1.0f / 16777216.0f);   // (0, 1)
    const float u2 = float(w.y >> 8) * (1.0f / 16777216.0f);            // [0, 1)
    const float r = sqrtf(-2.0f * __logf(u1));
    float s, c;
    __sincosf(6.283185307179586f * u2, &s, &c);
    return make_float2(r * c, r * s);
}

// one action component of the squashed head (SB3 SquashedDiagGaussianDistribution): pre-activations of the mu and log_std
// layers -> log_std clamped to [-20, 2], a = tanh(mu + exp(log_std) eps), act = clip(a + noise_std xi, -1, 1); lp is this
// component's log-prob of a without the -log(2 pi) / 2 constant: -eps^2 / 2 - log_std - log(1 - a^2 + 1e-6).  The accurate
// tanhf, not tanh.approx, and 1 - a^2 with one rounding (fma): the Jacobian term is sensitive near |a| -> 1, where a rounded
// a^2 alone moves log(1 - a^2 + 1e-6) by up to 0.06.  The log itself is __logf (lg2.approx: absolute error ~1e-7 over the
// whole range [1e-6, 1 + 1e-6]), 21 instructions per component fewer than logf
struct Squashed { float ls, act, lp; };
__device__ __forceinline__ Squashed squash(float mu, float ls_pre, float e, float xi, float noise_std) {
    Squashed s;
    s.ls = fminf(2.0f, fmaxf(-20.0f, ls_pre));
    const float act = tanhf(fmaf(expf(s.ls), e, mu));
    s.act = fminf(1.0f, fmaxf(-1.0f, fmaf(noise_std, xi, act)));
    s.lp = fmaf(-0.5f * e, e, -s.ls) - __logf(fmaf(-act, act, 1.0f) + 1e-6f);
    return s;
}

template <int HEAD>
__global__ void __launch_bounds__(THREADS, 2) policy_act_kernel(const __grid_constant__ PolicyArgs a) {
    extern __shared__ uint4 smem_raw[];
    unsigned char* smem = reinterpret_cast<unsigned char*>(smem_raw);
    {   // parameters: global (L2) -> shared, once per CTA
        const uint4* src = reinterpret_cast<const uint4*>(a.packed);
        for (int i = threadIdx.x; i < packed_bytes(HEAD) / 16; i += THREADS) smem_raw[i] = src[i];
    }
    __syncthreads();
    const uint2* w1 = reinterpret_cast<const uint2*>(smem + OFF_W1);
    const uint2* w2 = reinterpret_cast<const uint2*>(smem + OFF_W2);
    const uint2* w3 = reinterpret_cast<const uint2*>(smem + OFF_W3);
    const uint2* w4 = reinterpret_cast<const uint2*>(smem + OFF_W4);
    const float* bias = reinterpret_cast<const float*>(smem + OFF_B);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, g = lane >> 2, t = lane & 3;
    const long n_tiles = (a.n + TILE - 1) / TILE;
    // the observation rows of this thread's two environments (k = 2t, 2t + 1, 2t + 8, 2t + 9), already packed as the layer-1
    // A fragment; fetched one tile AHEAD: the loads of tile i + 1 are in flight while tile i runs through the network
    // (loaded at the top of the tile they cost a DRAM / L2 round trip per tile: long_scoreboard 2.7 per issue)
    auto load_obs = [&](long tile, unsigned (&a1)[4]) {
        const long r0 = tile * TILE + warp * 16 + g, r1 = r0 + 8;
        const bool ok0 = tile < n_tiles && r0 < a.n, ok1 = tile < n_tiles && r1 < a.n;
        float x[2][4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int k = 2 * t + (j & 1) + (j >> 1) * 8;
            const bool kv = k < a.obs_dim;
            x[0][j] = (kv && ok0) ? a.obs[(long)k * a.ld + r0] : 0.0f;
            x[1][j] = (kv && ok1) ? a.obs[(long)k * a.ld + r1] : 0.0f;
        }
        a1[0] = pack_bf16(x[0][0], x[0][1]); a1[1] = pack_bf16(x[1][0], x[1][1]);
        a1[2] = pack_bf16(x[0][2], x[0][3]); a1[3] = pack_bf16(x[1][2], x[1][3]);
    };
    unsigned a_next[4];
    load_obs(blockIdx.x, a_next);
    for (long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const long r0 = tile * TILE + warp * 16 + g, r1 = r0 + 8;
        const bool ok0 = r0 < a.n, ok1 = r1 < a.n;
        // ---- layer 1
        unsigned afr[8][4];
        {
            const unsigned a1[4] = {a_next[0], a_next[1], a_next[2], a_next[3]};
#if MVRL_POLICY_PREFETCH
            load_obs(tile + gridDim.x, a_next);
#endif
            float acc[16][4];
#pragma unroll
            for (int nt = 0; nt < 16; ++nt) {
                acc[nt][0] = acc[nt][1] = acc[nt][2] = acc[nt][3] = 0.0f;
                mma_bf16(acc[nt], a1, w1[nt * 32 + lane]);
            }
            activate_to_frags(acc, bias, t, afr);
        }
        // ---- layers 2 and 3 (128 x 128)
#pragma unroll 1
        for (int layer = 0; layer < 2; ++layer) {
            float acc[16][4];
            hidden_layer(layer == 0 ? w2 : w3, afr, lane, acc);
            activate_to_frags(acc, bias + (layer + 1) * H, t, afr);
        }
        // ---- head: 128 -> A (one n-tile), tanh mean, Gaussian sample
        float c4[4] = {0.0f, 0.0f, 0.0f, 0.0f};
#pragma unroll
        for (int kk = 0; kk < 8; ++kk) mma_bf16(c4, afr[kk], w4[kk * 32 + lane]);
        const int col = 2 * t;                       // this thread holds columns col, col + 1 of rows r0 (c4[0..1]) and r1 (c4[2..3])
        const float* b4 = bias + 3 * H;
        const float* sd = b4 + NOUT;
        float lp0 = 0.0f, lp1 = 0.0f;
        if constexpr (HEAD == HEAD_SQUASHED) {
            // second n-tile: the log_std layer (b4 = b_mu, sd = b_log_std)
            const uint2* wls = reinterpret_cast<const uint2*>(smem + OFF_WLS);
            float c5[4] = {0.0f, 0.0f, 0.0f, 0.0f};
#pragma unroll
            for (int kk = 0; kk < 8; ++kk) mma_bf16(c5, afr[kk], wls[kk * 32 + lane]);
            if (col < a.act_dim) {
                float2 e0 = make_float2(0.0f, 0.0f), e1 = e0, x0 = e0, x1 = e0;
                if (!a.deterministic) {
                    e0 = normal_pair(a.seed, a.env_id0 + (unsigned long long)r0, a.step, (unsigned)t);
                    e1 = normal_pair(a.seed, a.env_id0 + (unsigned long long)r1, a.step, (unsigned)t);
                    if (a.noise) {
                        x0 = normal_pair(a.seed, a.env_id0 + (unsigned long long)r0, a.step, (unsigned)t, STREAM_NOISE);
                        x1 = normal_pair(a.seed, a.env_id0 + (unsigned long long)r1, a.step, (unsigned)t, STREAM_NOISE);
                    }
                }
                const bool second = col + 1 < a.act_dim;
                const float m00 = c4[0] + b4[col], m01 = c4[1] + b4[col + 1], m10 = c4[2] + b4[col], m11 = c4[3] + b4[col + 1];
                const Squashed s00 = squash(m00, c5[0] + sd[col], e0.x, x0.x, a.noise_std[col]);
                const Squashed s01 = squash(m01, c5[1] + sd[col + 1], e0.y, x0.y, second ? a.noise_std[col + 1] : 0.0f);
                const Squashed s10 = squash(m10, c5[2] + sd[col], e1.x, x1.x, a.noise_std[col]);
                const Squashed s11 = squash(m11, c5[3] + sd[col + 1], e1.y, x1.y, second ? a.noise_std[col + 1] : 0.0f);
                lp0 = s00.lp + (second ? s01.lp : 0.0f);
                lp1 = s10.lp + (second ? s11.lp : 0.0f);
                if (ok0) {
                    a.act[(long)col * a.ld + r0] = s00.act;
                    if (second) a.act[(long)(col + 1) * a.ld + r0] = s01.act;
                    if (a.mean) { a.mean[(long)col * a.ld + r0] = m00; if (second) a.mean[(long)(col + 1) * a.ld + r0] = m01; }
                    if (a.log_std) { a.log_std[(long)col * a.ld + r0] = s00.ls; if (second) a.log_std[(long)(col + 1) * a.ld + r0] = s01.ls; }
                    if (a.eps) { a.eps[(long)col * a.ld + r0] = e0.x; if (second) a.eps[(long)(col + 1) * a.ld + r0] = e0.y; }
                }
                if (ok1) {
                    a.act[(long)col * a.ld + r1] = s10.act;
                    if (second) a.act[(long)(col + 1) * a.ld + r1] = s11.act;
                    if (a.mean) { a.mean[(long)col * a.ld + r1] = m10; if (second) a.mean[(long)(col + 1) * a.ld + r1] = m11; }
                    if (a.log_std) { a.log_std[(long)col * a.ld + r1] = s10.ls; if (second) a.log_std[(long)(col + 1) * a.ld + r1] = s11.ls; }
                    if (a.eps) { a.eps[(long)col * a.ld + r1] = e1.x; if (second) a.eps[(long)(col + 1) * a.ld + r1] = e1.y; }
                }
            }
        } else if (col < a.act_dim) {
            const float m00 = tanh_fast(c4[0] + b4[col]), m01 = tanh_fast(c4[1] + b4[col + 1]);
            const float m10 = tanh_fast(c4[2] + b4[col]), m11 = tanh_fast(c4[3] + b4[col + 1]);
            float2 e0 = make_float2(0.0f, 0.0f), e1 = e0;
            if (!a.deterministic) {
                e0 = normal_pair(a.seed, a.env_id0 + (unsigned long long)r0, a.step, (unsigned)t);
                e1 = normal_pair(a.seed, a.env_id0 + (unsigned long long)r1, a.step, (unsigned)t);
            }
            const bool second = col + 1 < a.act_dim;
            const float a00 = fminf(1.0f, fmaxf(-1.0f, fmaf(sd[col], e0.x, m00))), a01 = fminf(1.0f, fmaxf(-1.0f, fmaf(sd[col + 1], e0.y, m01)));
            const float a10 = fminf(1.0f, fmaxf(-1.0f, fmaf(sd[col], e1.x, m10))), a11 = fminf(1.0f, fmaxf(-1.0f, fmaf(sd[col + 1], e1.y, m11)));
            lp0 = -0.5f * (e0.x * e0.x + (second ? e0.y * e0.y : 0.0f));
            lp1 = -0.5f * (e1.x * e1.x + (second ? e1.y * e1.y : 0.0f));
            if (ok0) {
                a.act[(long)col * a.ld + r0] = a00;
                if (second) a.act[(long)(col + 1) * a.ld + r0] = a01;
                if (a.mean) { a.mean[(long)col * a.ld + r0] = m00; if (second) a.mean[(long)(col + 1) * a.ld + r0] = m01; }
                if (a.eps) { a.eps[(long)col * a.ld + r0] = e0.x; if (second) a.eps[(long)(col + 1) * a.ld + r0] = e0.y; }
            }
            if (ok1) {
                a.act[(long)col * a.ld + r1] = a10;
                if (second) a.act[(long)(col + 1) * a.ld + r1] = a11;
                if (a.mean) { a.mean[(long)col * a.ld + r1] = m10; if (second) a.mean[(long)(col + 1) * a.ld + r1] = m11; }
                if (a.eps) { a.eps[(long)col * a.ld + r1] = e1.x; if (second) a.eps[(long)(col + 1) * a.ld + r1] = e1.y; }
            }
        }
        // log-prob: sum over the action columns = over the four lanes of a quad
        lp0 += __shfl_xor_sync(0xffffffffu, lp0, 1); lp0 += __shfl_xor_sync(0xffffffffu, lp0, 2);
        lp1 += __shfl_xor_sync(0xffffffffu, lp1, 1); lp1 += __shfl_xor_sync(0xffffffffu, lp1, 2);
        if (a.logp != nullptr && t == 0) {
            if (ok0) a.logp[r0] = lp0 + a.logp_const;
            if (ok1) a.logp[r1] = lp1 + a.logp_const;
        }
#if !MVRL_POLICY_PREFETCH
        load_obs(tile + gridDim.x, a_next);
#endif
    }
}

unsigned short bf16_bits(float f) {   // round to nearest even, like __float2bfloat16_rn
    unsigned u;
    memcpy(&u, &f, 4);
    if ((u & 0x7fffffffu) > 0x7f800000u) return (unsigned short)((u >> 16) | 0x40);   // NaN
    u += 0x7fffu + ((u >> 16) & 1u);
    return (unsigned short)(u >> 16);
}

// W [N][K] (row = output unit, as torch.nn.Linear stores it) -> B fragments of mma.m16n8k16: for k-step kk, n-tile nt, lane
// (g = lane / 4, t = lane % 4): b0 = (W[8 nt + g][16 kk + 2t], +1), b1 = (W[8 nt + g][16 kk + 8 + 2t], +1); zeros outside N x K
void pack_b_fragments(const float* W, int N, int K, int n_tiles, int k_steps, unsigned char* dst) {
    unsigned* out = reinterpret_cast<unsigned*>(dst);
    auto at = [&](int n, int k) -> unsigned { return (n < N && k < K) ? bf16_bits(W[(size_t)n * K + k]) : 0u; };
    for (int kk = 0; kk < k_steps; ++kk)
        for (int nt = 0; nt < n_tiles; ++nt)
            for (int lane = 0; lane < 32; ++lane) {
                const int g = lane >> 2, t = lane & 3, n = 8 * nt + g, k0 = 16 * kk + 2 * t;
                const size_t i = ((size_t)(kk * n_tiles + nt) * 32 + lane) * 2;
                out[i] = at(n, k0) | (at(n, k0 + 1) << 16);
                out[i + 1] = at(n, k0 + 8) | (at(n, k0 + 9) << 16);
            }
}


// =====================================================================================================================
// tcgen05 version of the same network (the default): CTA tile = 128 environments = the 128 lanes of tensor memory.
// Per layer ONE thread issues tcgen05.mma (M = 128, N = 128, K = 16 per instruction, bf16 operands from shared memory
// through matrix descriptors, fp32 accumulator in TMEM), commits to an mbarrier; the four warps then read their lane
// quadrant of the accumulator with tcgen05.ld (thread = one environment's row), add the bias, apply GELU, pack to bf16 and
// store the row into the A operand of the next layer - in the canonical K-major core-matrix layout (8 rows x 16 bytes
// contiguous; LBO = 128 B between the K-chunks, SBO = (K / 8) * 128 B between 8-row groups; no swizzle), so the
// store of 8 consecutive lanes is one contiguous 128-byte line.  Weights sit in shared memory in the same layout
// (packed on the host), read by the tensor core ONCE per 128-row tile - the mma.sync version re-reads every B fragment
// for each 16 rows, 587 MB of shared-memory traffic per launch, its largest single cost.  2 CTAs per SM (106 KB of
// shared memory, 128 TMEM columns each): while one CTA's MMA runs, the other's epilogue keeps the MUFU / FMA pipes busy.
// (First version.  Now: ONE CTA per SM with GROUPS warpgroups, each running this protocol on its own tile - see the kernel.)
// Same bf16 operand rounding, same GELU code, same Philox streams as the mma.sync kernel (kept below it for A/B:
// MVRL_POLICY_MMA_SYNC=1); only the fp32 summation order inside the tensor core differs.
// =====================================================================================================================
namespace tc5 {

constexpr int TM = 128;                       // environments per tile
constexpr int HEAD_N = 16;                    // action columns padded to the smallest N of an M = 128 MMA
constexpr int OFF_W1 = 0;                     // [128 x 16]  bf16, canonical K-major
constexpr int OFF_W2 = OFF_W1 + H * KIN * 2;  // [128 x 128]
constexpr int OFF_W3 = OFF_W2 + H * H * 2;
constexpr int OFF_W4 = OFF_W3 + H * H * 2;    // [16 x 128]
constexpr int OFF_B = OFF_W4 + HEAD_N * H * 2;                  // float b1[128] b2[128] b3[128] b4[8] std[8]
#ifndef MVRL_POLICY_BIAS_MMA
#define MVRL_POLICY_BIAS_MMA 1   // hidden-layer biases added by the tensor core (one more K = 16 step per layer) instead of by the epilogue
#endif
constexpr bool BIAS_MMA = MVRL_POLICY_BIAS_MMA != 0;
constexpr int OFF_BIAS = OFF_B + (3 * H + 2 * NOUT) * 4;        // 3 x [128 x 16] bf16, canonical K-major: columns 0..2 = the bias split into three bf16 terms
constexpr int OFF_ONES = OFF_BIAS + (BIAS_MMA ? 3 * H * KIN * 2 : 0);   // [128 x 16] bf16, canonical K-major: columns 0..2 = 1
constexpr int PARAM_BYTES = OFF_ONES + (BIAS_MMA ? TM * KIN * 2 : 0);
constexpr int OFF_A = (PARAM_BYTES + 127) / 128 * 128;          // activations [128 x 128] bf16 per warpgroup, canonical K-major
constexpr int A_BYTES = TM * H * 2;
#ifndef MVRL_POLICY_GROUPS
#define MVRL_POLICY_GROUPS 4     // warpgroups (= tiles in flight) per CTA; one CTA per SM
#endif
constexpr int GROUPS = MVRL_POLICY_GROUPS;
constexpr int SMEM_BYTES = OFF_A + GROUPS * A_BYTES;
constexpr int TMEM_COLS = GROUPS * H <= 128 ? 128 : (GROUPS * H <= 256 ? 256 : 512);
static_assert(GROUPS >= 1 && GROUPS * H <= 512 && SMEM_BYTES <= 227 * 1024, "warpgroups per CTA limited by TMEM columns and shared memory");
static_assert(PARAM_BYTES % 16 == 0, "parameter block is copied with 16-byte accesses");

__device__ __forceinline__ unsigned long long smem_desc(unsigned addr, unsigned lbo, unsigned sbo) {
    // SM100 shared-memory matrix descriptor: start address, leading / stride byte offsets (all >> 4), version 1, no swizzle
    return (unsigned long long)((addr & 0x3FFFFu) >> 4) | ((unsigned long long)(lbo >> 4) << 16) | ((unsigned long long)(sbo >> 4) << 32) |
           (1ull << 46);
}
// instruction descriptor of kind::f16: fp32 accumulator, bf16 A and B, both K-major, N >> 3 at bit 17, M >> 4 at bit 24
__host__ __device__ constexpr unsigned instr_desc(int m, int n) {
    return (1u << 4) | (1u << 7) | (1u << 10) | ((unsigned)(n >> 3) << 17) | ((unsigned)(m >> 4) << 24);
}
__device__ __forceinline__ void mma_ss(unsigned d_tmem, unsigned long long a_desc, unsigned long long b_desc, unsigned idesc, unsigned accumulate) {
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
                 "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, {%5, %5, %5, %5}, p;\n\t}"
                 ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate), "r"(0u) : "memory");
}
__device__ __forceinline__ void tmem_ld32(unsigned taddr, unsigned (&v)[32]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x32.b32 "
                 "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]), "=r"(v[10]),
                   "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]),
                   "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]),
                   "=r"(v[31])
                 : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tmem_ld16(unsigned taddr, unsigned (&v)[16]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]), "=r"(v[10]),
                   "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
                 : "r"(taddr) : "memory");
}

#ifndef MVRL_POLICY_LDTM_PIPE
#define MVRL_POLICY_LDTM_PIPE 1
#endif
#ifndef MVRL_POLICY_PINGPONG
#define MVRL_POLICY_PINGPONG 1   // the two pairs of tile groups take turns in the epilogue (see the kernel)
#endif
#ifndef MVRL_POLICY_SPLIT
#define MVRL_POLICY_SPLIT 1      // threads per environment row in the epilogues (1 or 2); 2 (8 warps per tile, 64 columns each, 64 registers) measured slower: 34.0 vs 31.9 us, and 28.8 vs 24.4 us with the turn schedule
#endif
constexpr int SPLIT = MVRL_POLICY_SPLIT;
constexpr int GT = TM * SPLIT;   // threads of a tile group
static_assert(SPLIT == 1 || SPLIT == 2, "a TMEM lane quadrant is reachable from warps w and w + 4 only");
static_assert(GT * GROUPS <= 1024, "CTA size");

template <int HEAD>
__global__ void __launch_bounds__(GT * GROUPS, 1) policy_act_tc5_kernel(const __grid_constant__ PolicyArgs a) {
    extern __shared__ __align__(128) unsigned char smem[];
    __shared__ __align__(8) unsigned long long mma_bars[GROUPS];
    __shared__ __align__(8) unsigned long long weights_bar;
    __shared__ float lp_part[GROUPS][TM];
    __shared__ unsigned tmem_base_slot;
    // a tile group (SPLIT x 128 threads: thread = one environment's row = one TMEM lane, SPLIT threads share a row's columns)
    // owns one tile at a time: its own A operand buffer, accumulator columns, mbarrier and named barrier; the GROUPS groups
    // of the CTA share only the weights and run out of phase
    const int group = threadIdx.x / GT, gt = threadIdx.x % GT, row = gt % TM, half = gt / TM;
    const unsigned bar = (unsigned)__cvta_generic_to_shared(&mma_bars[group]);
    const unsigned wbar = (unsigned)__cvta_generic_to_shared(&weights_bar);
    if (gt == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar));
        if (group == 0) asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(wbar));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (threadIdx.x < 32) {   // 128 TMEM columns per group: the fp32 accumulator of one 128 x 128 layer (the head reuses the first 16)
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"((unsigned)__cvta_generic_to_shared(&tmem_base_slot)), "n"(TMEM_COLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    // parameters: global (L2) -> shared, once per CTA, as ONE bulk copy (73 KB) that lands while the first observations are
    // fetched and packed; every thread waits for it once, before its group's first MMA / bias read.  (Copied by the threads
    // with 16-byte loads it was 14 % of the kernel's stall samples: nine dependent L2 round trips per thread.)
    if (threadIdx.x == 0) {
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(wbar), "n"(PARAM_BYTES) : "memory");
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                     ::"r"((unsigned)__cvta_generic_to_shared(smem)), "l"(a.packed), "n"(PARAM_BYTES), "r"(wbar) : "memory");
    }
    const unsigned tmem_all = tmem_base_slot;
    const unsigned tmem_d = tmem_all + (unsigned)(group * H);
    const unsigned tmem_row = tmem_d + ((unsigned)(row & ~31) << 16);   // this warp's lane quadrant (warps w and w + 4 of a group share one)
    const unsigned smem_base = (unsigned)__cvta_generic_to_shared(smem);
    const unsigned a_addr = smem_base + OFF_A + group * A_BYTES;
    const float* bias = reinterpret_cast<const float*>(smem + OFF_B);
    unsigned char* a_buf = smem + OFF_A + group * A_BYTES;
    unsigned char* a_row16 = a_buf + (row >> 3) * (KIN / 8 * 128) + (row & 7) * 16;   // this thread's row, K = 16 layout (SBO 256)
    unsigned char* a_row128 = a_buf + (row >> 3) * (H / 8 * 128) + (row & 7) * 16;    // K = 128 layout (SBO 2048)
    unsigned parity = 0;
    // one layer's MMAs: D[128 x N] (+)= A[128 x K] B[N x K]^T, K / 16 instructions, then commit -> mbarrier
    auto issue_layer = [&](int w_off, int K, int N, int bias_off) {
        const unsigned sbo = (unsigned)(K / 8) * 128u;
        const unsigned long long ad = smem_desc(a_addr, 128u, sbo), bd = smem_desc(smem_base + w_off, 128u, sbo);
        const unsigned idesc = instr_desc(TM, N);
        for (int j = 0; j < K / 16; ++j)      // a K = 16 step is two 128-byte core-matrix columns: 256 bytes = 16 descriptor units
            mma_ss(tmem_d, ad + (unsigned long long)(16 * j), bd + (unsigned long long)(16 * j), idesc, j > 0 ? 1u : 0u);
        if (BIAS_MMA && bias_off >= 0)   // + 1 b^T: one more K = 16 step, A = the constant ones block, B = the bias as three bf16 terms (their sum is the fp32 bias)
            mma_ss(tmem_d, smem_desc(smem_base + OFF_ONES, 128u, 256u), smem_desc(smem_base + bias_off, 128u, 256u), idesc, 1u);
        asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
    };
    auto wait_layer = [&]() {
        unsigned done = 0;
        while (!done)
            asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2; selp.u32 %0, 1, 0, p; }"
                         : "=r"(done) : "r"(bar), "r"(parity) : "memory");
        parity ^= 1u;
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    };
    // hand the freshly written A operand (and the drained accumulator) over to the MMA-issuing thread
    auto publish = [&]() {
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        asm volatile("bar.sync %0, %1;" ::"r"(group + 1), "n"(GT) : "memory");   // this group only
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    };
    constexpr int XW = KIN / SPLIT;           // observation components per thread: k in [half * XW, half * XW + XW)
    // tiles are dealt out to the SMs first (tile t -> CTA t % gridDim.x), then to the groups of a CTA: every SM gets the same
    // number of tiles +- 1 (131 072 envs: 7 or 6 per SM; dealt to groups first, 108 SMs had 8 and 40 SMs had 4)
    const long n_tiles = (a.n + TM - 1) / TM;
    const long tile_step = (long)gridDim.x * GROUPS;
    const long first_tile = (long)blockIdx.x + (long)gridDim.x * group;
    auto load_obs = [&](long tile, float (&x)[XW]) {
        const long r = tile * TM + row;
        const bool ok = tile < n_tiles && r < a.n;
#pragma unroll
        for (int k = 0; k < XW; ++k) x[k] = (ok && half * XW + k < a.obs_dim) ? a.obs[(long)(half * XW + k) * a.ld + r] : 0.0f;
    };
    float x[XW];
    load_obs(first_tile, x);
    {   // the parameter block has landed (async proxy -> visible to the tensor core and, after this wait, to this thread)
        unsigned done = 0;
        while (!done)
            asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2; selp.u32 %0, 1, 0, p; }"
                         : "=r"(done) : "r"(wbar), "r"(0u) : "memory");
    }
    long pending_r = -1;        // SPLIT == 2: the log-prob of the previous tile waits for the other half's partial sum
    float pending_lp = 0.0f;
    // PING-PONG.  Left alone, the four groups of a CTA run in lock step: they share the XU pipe fairly, so their epilogues
    // end together, their MMAs are issued together and queue on the one tensor core (each group then waits ~2000 cycles for
    // 576 cycles of MMA), and the XU pipe idles meanwhile - a third of a tile's 21.5 k cycles was MMA wait (clock64 trace,
    // tools/exp/actor_trace.py).  So the groups are split into two pairs that take turns: a pair enters a hidden-layer
    // epilogue only when the other pair has left its own (two named barriers, bar.sync by the pair that waits, bar.arrive by
    // the pair that leaves) - while one pair keeps the XU pipe busy, the other pair's MMAs run and complete.  Every group
    // goes through the same number of turns; a group without a tile in an iteration just passes the turn on.  (Also measured:
    // single groups in round-robin order with at most 1 / 2 / 3 in the epilogue at a time, by counters polled in shared memory:
    // 29.6 / 24.8 / 25.3 us against 24.2 us for this pair scheme - tools/exp/r2ab.sh.  Named barriers cannot count: a group
    // that runs two epilogues ahead of its waiter completes a barrier phase on its own, and the CTA dead-locks.)
    constexpr bool PINGPONG = (MVRL_POLICY_PINGPONG != 0) && GROUPS == 4;
    const int pair = group >> 1;
    const long tiles_cta = (long)blockIdx.x < n_tiles ? (n_tiles - 1 - (long)blockIdx.x) / (long)gridDim.x + 1 : 0;   // tiles dealt to this CTA
    const long iters = PINGPONG ? (tiles_cta + GROUPS - 1) / GROUPS : (tiles_cta > group ? (tiles_cta - group + GROUPS - 1) / GROUPS : 0);
    long turn = 0;
    const long turns = 3 * iters;
    auto enter_epilogue = [&]() {
        if (PINGPONG) asm volatile("bar.sync %0, %1;" ::"r"(5 + pair), "n"(2 * GT * 2) : "memory");
    };
    auto leave_epilogue = [&]() {
        if (PINGPONG) {
            ++turn;
            if (!(pair == 1 && turn == turns)) asm volatile("bar.arrive %0, %1;" ::"r"(5 + (pair ^ 1)), "n"(2 * GT * 2) : "memory");
        }
    };
    if (PINGPONG && pair == 1 && turns > 0) asm volatile("bar.arrive %0, %1;" ::"r"(5), "n"(2 * GT * 2) : "memory");   // the first turn is pair 0's
    for (long it = 0; it < iters; ++it) {
        const long tile = first_tile + it * tile_step;
        if (tile >= n_tiles) {      // (ping-pong only) no tile in this iteration: pass the three turns on
            for (int layer = 0; layer < 3; ++layer) { enter_epilogue(); leave_epilogue(); }
            continue;
        }
        const long r = tile * TM + row;
        const bool ok = r < a.n;
        // ---- this environment's observation row as the K = 16 A operand of layer 1
#pragma unroll
        for (int c = 0; c < XW / 8; ++c)
            *reinterpret_cast<uint4*>(a_row16 + (half * (XW / 8) + c) * 128) = make_uint4(pack_bf16(x[8 * c], x[8 * c + 1]), pack_bf16(x[8 * c + 2], x[8 * c + 3]),
                                                                                         pack_bf16(x[8 * c + 4], x[8 * c + 5]), pack_bf16(x[8 * c + 6], x[8 * c + 7]));
        publish();
        if (gt == 0) issue_layer(OFF_W1, KIN, H, OFF_BIAS);
        if (SPLIT == 2 && half == 0 && pending_r >= 0) {      // the barrier above made the other half's partial visible
            a.logp[pending_r] = pending_lp + lp_part[group][row] + a.logp_const;
            pending_r = -1;
        }
        load_obs(tile + tile_step, x);            // the next tile's observations travel while this tile runs through the network
        // the Gaussian noise of this environment's action pairs does not depend on the network: one Philox block + Box-Muller
        // per MMA in flight, computed in the shadow of the tensor core instead of after the head (29.2 -> 25.7 us)
        float2 eps[NOUT / 2], xi[NOUT / 2];   // xi: the squashed head's action noise
#pragma unroll
        for (int pr = 0; pr < NOUT / 2; ++pr) eps[pr] = xi[pr] = make_float2(0.0f, 0.0f);
        auto draw = [&](int pr) {
            if (!a.deterministic && 2 * pr < a.act_dim && (pr % SPLIT) == half) {
                eps[pr] = normal_pair(a.seed, a.env_id0 + (unsigned long long)r, a.step, (unsigned)pr);
                if (HEAD == HEAD_SQUASHED && a.noise) xi[pr] = normal_pair(a.seed, a.env_id0 + (unsigned long long)r, a.step, (unsigned)pr, STREAM_NOISE);
            }
        };
        draw(0);
#pragma unroll
        for (int layer = 0; layer < 3; ++layer) {
            wait_layer();
            enter_epilogue();
            const float* b = bias + layer * H;
            // (free-running groups did not profit from the double-buffered tcgen05.ld below, 26.1 vs 25.7 us - other warps hid the
            // latency; with the turn schedule it is worth 5 %: 24.05 -> 22.85 us)
            // ---- epilogue of hidden layer `layer`: accumulator row -> bias + GELU -> bf16 -> A operand of the next layer
#if MVRL_POLICY_LDTM_PIPE
            // 16-column chunks, double-buffered: the tcgen05.ld of chunk k + 1 is in flight while chunk k goes through the GELU
            // (tcgen05.wait::ld waits for every outstanding load of the thread, so it comes AFTER the arithmetic of chunk k).
            // With the turn schedule only two warps per scheduler are in an epilogue, and nothing else hides the TMEM read latency.
            {
                constexpr int NCH = H / SPLIT / 16;
                const int cbase = half * (H / SPLIT);
                unsigned v[2][16];
                tmem_ld16(tmem_row + (unsigned)cbase, v[0]);
                asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
                for (int ch = 0; ch < NCH; ++ch) {
                    const int c0 = cbase + 16 * ch;
                    if (ch + 1 < NCH) tmem_ld16(tmem_row + (unsigned)(c0 + 16), v[(ch + 1) & 1]);
                    const unsigned (&w)[16] = v[ch & 1];
#pragma unroll
                    for (int q = 0; q < 2; ++q) {     // 8 columns = one 16-byte chunk of the row
                        unsigned pk[4];
#pragma unroll
                        for (int e = 0; e < 4; ++e) {
                            const int col = c0 + 8 * q + 2 * e;
                            if (BIAS_MMA) pk[e] = gelu2x_pack2(__uint_as_float(w[8 * q + 2 * e]), __uint_as_float(w[8 * q + 2 * e + 1]));
                            else pk[e] = gelu_pack2(__uint_as_float(w[8 * q + 2 * e]), __uint_as_float(w[8 * q + 2 * e + 1]), *reinterpret_cast<const float2*>(b + col));
                        }
                        *reinterpret_cast<uint4*>(a_row128 + ((c0 >> 3) + q) * 128) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
                    }
                    if (ch + 1 < NCH) asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
                }
            }
#else
#pragma unroll 1
            for (int c0 = half * (H / SPLIT); c0 < (half + 1) * (H / SPLIT); c0 += 32) {
                unsigned v[32];
                tmem_ld32(tmem_row + (unsigned)c0, v);
                asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
                for (int q = 0; q < 4; ++q) {     // 8 columns = one 16-byte chunk of the row
                    unsigned pk[4];
#pragma unroll
                    for (int e = 0; e < 4; ++e) {
                        const int col = c0 + 8 * q + 2 * e;
                        if (BIAS_MMA) pk[e] = gelu2x_pack2(__uint_as_float(v[8 * q + 2 * e]), __uint_as_float(v[8 * q + 2 * e + 1]));
                        else pk[e] = gelu_pack2(__uint_as_float(v[8 * q + 2 * e]), __uint_as_float(v[8 * q + 2 * e + 1]), *reinterpret_cast<const float2*>(b + col));
                    }
                    *reinterpret_cast<uint4*>(a_row128 + ((c0 >> 3) + q) * 128) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
                }
            }
#endif
            leave_epilogue();
            publish();
            if (gt == 0) {
                if (layer < 2) issue_layer(layer == 0 ? OFF_W2 : OFF_W3, H, H, OFF_BIAS + (layer + 1) * H * KIN * 2);
                else issue_layer(OFF_W4, H, HEAD_N, -1);     // the six head biases are added in fp32 by the epilogue
            }
            draw(layer + 1);
        }
        // ---- head: 128 -> A columns of this environment's row, tanh mean, Gaussian sample, log-prob; the action pairs
        // (2 pr, 2 pr + 1) of a row are dealt out to its SPLIT threads
        wait_layer();
        unsigned hv[16];
        tmem_ld16(tmem_row, hv);
        asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
        const float* b4 = bias + 3 * H;
        const float* sd = b4 + NOUT;
        float lp = 0.0f;
#pragma unroll
        for (int pr = 0; pr < NOUT / 2; ++pr) {
            const int col = 2 * pr;
            if (HEAD == HEAD_SQUASHED && col < a.act_dim && (pr % SPLIT) == half) {
                // mu in columns 0..7, the log_std layer in columns 8..15 of the same accumulator (b4 = b_mu, sd = b_log_std)
                const bool second = col + 1 < a.act_dim;
                const float m0 = __uint_as_float(hv[col]) + b4[col], m1 = __uint_as_float(hv[col + 1]) + b4[col + 1];
                const float2 e = eps[pr], x = xi[pr];
                const Squashed s0 = squash(m0, __uint_as_float(hv[NOUT + col]) + sd[col], e.x, x.x, a.noise_std[col]);
                const Squashed s1 = squash(m1, __uint_as_float(hv[NOUT + col + 1]) + sd[col + 1], e.y, x.y, a.noise_std[col + 1]);
                lp += s0.lp + (second ? s1.lp : 0.0f);
                if (ok) {
                    a.act[(long)col * a.ld + r] = s0.act;
                    if (second) a.act[(long)(col + 1) * a.ld + r] = s1.act;
                    if (a.mean) { a.mean[(long)col * a.ld + r] = m0; if (second) a.mean[(long)(col + 1) * a.ld + r] = m1; }
                    if (a.log_std) { a.log_std[(long)col * a.ld + r] = s0.ls; if (second) a.log_std[(long)(col + 1) * a.ld + r] = s1.ls; }
                    if (a.eps) { a.eps[(long)col * a.ld + r] = e.x; if (second) a.eps[(long)(col + 1) * a.ld + r] = e.y; }
                }
            } else if (HEAD == HEAD_FIXED && col < a.act_dim && (pr % SPLIT) == half) {
                const bool second = col + 1 < a.act_dim;
                const float m0 = tanh_fast(__uint_as_float(hv[col]) + b4[col]), m1 = tanh_fast(__uint_as_float(hv[col + 1]) + b4[col + 1]);
                const float2 e = eps[pr];
                const float a0 = fminf(1.0f, fmaxf(-1.0f, fmaf(sd[col], e.x, m0))), a1 = fminf(1.0f, fmaxf(-1.0f, fmaf(sd[col + 1], e.y, m1)));
                lp += -0.5f * (e.x * e.x + (second ? e.y * e.y : 0.0f));
                if (ok) {
                    a.act[(long)col * a.ld + r] = a0;
                    if (second) a.act[(long)(col + 1) * a.ld + r] = a1;
                    if (a.mean) { a.mean[(long)col * a.ld + r] = m0; if (second) a.mean[(long)(col + 1) * a.ld + r] = m1; }
                    if (a.eps) { a.eps[(long)col * a.ld + r] = e.x; if (second) a.eps[(long)(col + 1) * a.ld + r] = e.y; }
                }
            }
        }
        if (SPLIT == 1) {
            if (a.logp != nullptr && ok) a.logp[r] = lp + a.logp_const;
        } else if (half == 1) {
            lp_part[group][row] = lp;
        } else if (a.logp != nullptr && ok) {
            pending_r = r; pending_lp = lp;
        }
        // the next tile's first publish() orders these accumulator reads before the next layer-1 MMA overwrites TMEM
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (SPLIT == 2 && half == 0 && pending_r >= 0) a.logp[pending_r] = pending_lp + lp_part[group][row] + a.logp_const;
    if (threadIdx.x < 32) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_all), "n"(TMEM_COLS) : "memory");
}

// W [N][K] (row = output unit, K contiguous: torch.nn.Linear) -> canonical K-major core-matrix order, zero padded to Np x Kp:
// element (n, k) at bf16 index ((n / 8) * (Kp / 8) + k / 8) * 64 + (n % 8) * 8 + k % 8
void pack_canonical(const float* W, int N, int K, int Np, int Kp, unsigned char* dst) {
    unsigned short* out = reinterpret_cast<unsigned short*>(dst);
    for (int n = 0; n < Np; ++n)
        for (int k = 0; k < Kp; ++k)
            out[((size_t)(n / 8) * (Kp / 8) + k / 8) * 64 + (n % 8) * 8 + k % 8] = (n < N && k < K) ? bf16_bits(W[(size_t)n * K + k]) : (unsigned short)0;
}

}  // namespace tc5

}  // namespace

struct MvrlPolicy {
    int device, obs_dim, act_dim, sm_count;
    int head;                // MVRL_POLICY_HEAD_*: the kernel instantiation this handle launches
    unsigned char* packed;   // device: B fragments of the mma.sync kernel
    unsigned char* packed5;  // device: canonical K-major matrices of the tcgen05 kernel
    bool mma_sync;           // MVRL_POLICY_MMA_SYNC=1: the warp-level mma.sync kernel instead of tcgen05
    bool has_weights;
    float logp_const;        // fixed head: -sum(log_std); squashed head: -act_dim log(2 pi) / 2
    bool noise;              // squashed head: action noise on
    float noise_std[NOUT];
};

extern "C" MVRL_API int mvrl_policy_create_head(MvrlPolicy** out, int device, int obs_dim, int act_dim, int head) {
    if (!out) return mvrl_fail(MVRL_EINVAL, "mvrl_policy_create: null output");
    if (obs_dim < 1 || obs_dim > KIN || act_dim < 1 || act_dim > NOUT)
        return mvrl_fail(MVRL_EINVAL, "mvrl_policy_create: obs_dim must be 1..%d and act_dim 1..%d (got %d, %d)", KIN, NOUT, obs_dim, act_dim);
    if (head != HEAD_FIXED && head != HEAD_SQUASHED)
        return mvrl_fail(MVRL_EINVAL, "mvrl_policy_create_head: unknown head %d (MVRL_POLICY_HEAD_FIXED_STD or MVRL_POLICY_HEAD_SQUASHED)", head);
    { const int rc = mvrl_require_device(device); if (rc != MVRL_OK) return rc; }
    MVRL_ON_DEVICE(device);
    MvrlPolicy* h = new (std::nothrow) MvrlPolicy();
    if (!h) return mvrl_fail(MVRL_EINVAL, "out of host memory");
    h->device = device; h->obs_dim = obs_dim; h->act_dim = act_dim; h->has_weights = false; h->logp_const = 0.f; h->packed = nullptr; h->packed5 = nullptr;
    h->head = head; h->noise = false;
    for (int k = 0; k < NOUT; ++k) h->noise_std[k] = 0.0f;
    { const char* e = getenv("MVRL_POLICY_MMA_SYNC"); h->mma_sync = (e && e[0] == '1'); }
    h->sm_count = 148;
    { int v = 0; if (cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, device) == cudaSuccess && v > 0) h->sm_count = v; else cudaGetLastError(); }
    cudaError_t e = cudaMalloc(&h->packed, packed_bytes(head));
    if (e == cudaSuccess) e = cudaMalloc(&h->packed5, tc5::PARAM_BYTES);
    if (head == HEAD_FIXED) {
        if (e == cudaSuccess) e = cudaFuncSetAttribute(policy_act_kernel<HEAD_FIXED>, cudaFuncAttributeMaxDynamicSharedMemorySize, PACKED_BYTES);
        if (e == cudaSuccess) e = cudaFuncSetAttribute(tc5::policy_act_tc5_kernel<HEAD_FIXED>, cudaFuncAttributeMaxDynamicSharedMemorySize, tc5::SMEM_BYTES);
    } else {
        if (e == cudaSuccess) e = cudaFuncSetAttribute(policy_act_kernel<HEAD_SQUASHED>, cudaFuncAttributeMaxDynamicSharedMemorySize, PACKED_BYTES_SQUASHED);
        if (e == cudaSuccess) e = cudaFuncSetAttribute(tc5::policy_act_tc5_kernel<HEAD_SQUASHED>, cudaFuncAttributeMaxDynamicSharedMemorySize, tc5::SMEM_BYTES);
    }
    if (e != cudaSuccess) {
        if (h->packed) cudaFree(h->packed);
        if (h->packed5) cudaFree(h->packed5);
        delete h;
        return mvrl_fail(MVRL_ECUDA, "mvrl_policy_create: %s", cudaGetErrorString(e));
    }
    *out = h;
    return MVRL_OK;
}

extern "C" MVRL_API int mvrl_policy_create(MvrlPolicy** out, int device, int obs_dim, int act_dim) {
    return mvrl_policy_create_head(out, device, obs_dim, act_dim, HEAD_FIXED);
}

extern "C" MVRL_API int mvrl_policy_destroy(MvrlPolicy* h) {
    if (!h) return MVRL_OK;
    { MvrlDeviceGuard guard(h->device); cudaFree(h->packed); cudaFree(h->packed5); }
    delete h;
    return MVRL_OK;
}

// Both kernels' parameter blocks from host arrays in torch.nn.Linear layout; synchronises.  W4 [act_dim][H] is the first head
// layer (fixed: the mean, squashed: mu), Wls [act_dim][H] the squashed head's log_std layer (NULL for the fixed head); v0 / v1
// [act_dim] go to the b4 / std slots of the fp32 block (fixed: b4, exp(log_std); squashed: b_mu, b_log_std).
static int upload_weights(MvrlPolicy* h, const float* W1, const float* b1, const float* W2, const float* b2, const float* W3, const float* b3,
                          const float* W4, const float* Wls, const float* v0, const float* v1) {
    const int pbytes = packed_bytes(h->head);
    std::vector<unsigned char> buf(pbytes, 0);
    pack_b_fragments(W1, H, h->obs_dim, 16, 1, buf.data() + OFF_W1);
    pack_b_fragments(W2, H, H, 16, 8, buf.data() + OFF_W2);
    pack_b_fragments(W3, H, H, 16, 8, buf.data() + OFF_W3);
    pack_b_fragments(W4, h->act_dim, H, 1, 8, buf.data() + OFF_W4);
    if (Wls) pack_b_fragments(Wls, h->act_dim, H, 1, 8, buf.data() + OFF_WLS);
    float* fb = reinterpret_cast<float*>(buf.data() + OFF_B);
    memcpy(fb, b1, H * 4); memcpy(fb + H, b2, H * 4); memcpy(fb + 2 * H, b3, H * 4);
    for (int k = 0; k < h->act_dim; ++k) { fb[3 * H + k] = v0[k]; fb[3 * H + NOUT + k] = v1[k]; }
    MVRL_ON_DEVICE(h->device);
    MVRL_CUDA(cudaMemcpy(h->packed, buf.data(), pbytes, cudaMemcpyHostToDevice));
    std::vector<unsigned char> buf5(tc5::PARAM_BYTES, 0);
    tc5::pack_canonical(W1, H, h->obs_dim, H, KIN, buf5.data() + tc5::OFF_W1);
    {   // the hidden activations are stored doubled (gelu2x_pack2): the layers that read them get half the weights.  The head
        // block is [16 x 128]: the first head layer in rows 0..act_dim-1, the squashed head's log_std layer in rows 8..
        const float in_scale = tc5::BIAS_MMA ? 0.5f : 1.0f;
        std::vector<float> w2((size_t)H * H), w3((size_t)H * H), w4((size_t)tc5::HEAD_N * H, 0.0f);
        for (size_t i = 0; i < w2.size(); ++i) { w2[i] = in_scale * W2[i]; w3[i] = in_scale * W3[i]; }
        for (size_t i = 0; i < (size_t)h->act_dim * H; ++i) w4[i] = in_scale * W4[i];
        if (Wls)
            for (size_t i = 0; i < (size_t)h->act_dim * H; ++i) w4[(size_t)NOUT * H + i] = in_scale * Wls[i];
        tc5::pack_canonical(w2.data(), H, H, H, H, buf5.data() + tc5::OFF_W2);
        tc5::pack_canonical(w3.data(), H, H, H, H, buf5.data() + tc5::OFF_W3);
        tc5::pack_canonical(w4.data(), tc5::HEAD_N, H, tc5::HEAD_N, H, buf5.data() + tc5::OFF_W4);
    }
    memcpy(buf5.data() + tc5::OFF_B, fb, (3 * H + 2 * NOUT) * 4);
    if (tc5::BIAS_MMA) {   // bias blocks: b = t0 + t1 + t2 with every term a bf16 (24 mantissa bits in all: the fp32 bias), and the ones block
        const float* bs[3] = {b1, b2, b3};
        std::vector<float> terms((size_t)H * 3), ones((size_t)tc5::TM * 3, 1.0f);
        auto bf16_value = [](float f) { unsigned u = (unsigned)bf16_bits(f) << 16; float r; memcpy(&r, &u, 4); return r; };
        for (int l = 0; l < 3; ++l) {
            for (int n = 0; n < H; ++n) {
                float rest = bs[l][n];
                for (int t = 0; t < 3; ++t) { const float q = bf16_value(rest); terms[(size_t)n * 3 + t] = q; rest -= q; }
            }
            tc5::pack_canonical(terms.data(), H, 3, H, KIN, buf5.data() + tc5::OFF_BIAS + l * H * KIN * 2);
        }
        tc5::pack_canonical(ones.data(), tc5::TM, 3, tc5::TM, KIN, buf5.data() + tc5::OFF_ONES);
    }
    MVRL_CUDA(cudaMemcpy(h->packed5, buf5.data(), tc5::PARAM_BYTES, cudaMemcpyHostToDevice));
    h->has_weights = true;
    return MVRL_OK;
}

extern "C" MVRL_API int mvrl_policy_set_weights(MvrlPolicy* h, const float* W1, const float* b1, const float* W2, const float* b2,
                                                const float* W3, const float* b3, const float* W4, const float* b4, const float* log_std) {
    if (!h || !W1 || !b1 || !W2 || !b2 || !W3 || !b3 || !W4 || !b4 || !log_std) return mvrl_fail(MVRL_EINVAL, "mvrl_policy_set_weights: null argument");
    if (h->head != HEAD_FIXED) return mvrl_fail(MVRL_EINVAL, "mvrl_policy_set_weights: the handle has the squashed head (mvrl_policy_set_weights_squashed)");
    float sd[NOUT];
    double lsum = 0;
    for (int k = 0; k < h->act_dim; ++k) { sd[k] = expf(log_std[k]); lsum += log_std[k]; }
    const int rc = upload_weights(h, W1, b1, W2, b2, W3, b3, W4, nullptr, b4, sd);
    if (rc == MVRL_OK) h->logp_const = (float)(-lsum);
    return rc;
}

extern "C" MVRL_API int mvrl_policy_set_weights_squashed(MvrlPolicy* h, const float* W1, const float* b1, const float* W2, const float* b2,
                                                         const float* W3, const float* b3, const float* W_mu, const float* b_mu,
                                                         const float* W_log_std, const float* b_log_std, const float* noise_std) {
    if (!h || !W1 || !b1 || !W2 || !b2 || !W3 || !b3 || !W_mu || !b_mu || !W_log_std || !b_log_std)
        return mvrl_fail(MVRL_EINVAL, "mvrl_policy_set_weights_squashed: null argument");
    if (h->head != HEAD_SQUASHED) return mvrl_fail(MVRL_EINVAL, "mvrl_policy_set_weights_squashed: the handle has the fixed-std head (mvrl_policy_set_weights)");
    if (noise_std)
        for (int k = 0; k < h->act_dim; ++k)
            if (!(noise_std[k] >= 0.0f && noise_std[k] < INFINITY))
                return mvrl_fail(MVRL_EINVAL, "mvrl_policy_set_weights_squashed: noise_std[%d] = %g is not a finite value >= 0", k, (double)noise_std[k]);
    const int rc = upload_weights(h, W1, b1, W2, b2, W3, b3, W_mu, W_log_std, b_mu, b_log_std);
    if (rc != MVRL_OK) return rc;
    h->logp_const = (float)(-0.5 * h->act_dim * log(2.0 * M_PI));
    h->noise = noise_std != nullptr;
    for (int k = 0; k < NOUT; ++k) h->noise_std[k] = (noise_std && k < h->act_dim) ? noise_std[k] : 0.0f;
    return MVRL_OK;
}

extern "C" MVRL_API int mvrl_policy_act_ex(MvrlPolicy* h, int64_t n, int64_t ld, const float* obs, float* act, float* logp, float* mean,
                                           float* log_std, float* eps, uint64_t seed, uint64_t env_id0, uint32_t step, int deterministic,
                                           mvrl_stream_t stream) {
    if (!h || !obs || !act) return mvrl_fail(MVRL_EINVAL, "mvrl_policy_act: null argument");
    if (n < 0 || ld < n) return mvrl_fail(MVRL_EINVAL, "mvrl_policy_act: need 0 <= n <= ld");
    if (log_std && h->head != HEAD_SQUASHED) return mvrl_fail(MVRL_EINVAL, "mvrl_policy_act_ex: log_std is an output of the squashed head only");
    if (!h->has_weights) return mvrl_fail(MVRL_EINVAL, "mvrl_policy_act: call mvrl_policy_set_weights first");
    if (n == 0) return MVRL_OK;
    MVRL_ON_DEVICE(h->device);
    PolicyArgs a;
    a.packed = h->packed; a.n = n; a.ld = ld; a.obs = obs; a.act = act; a.logp = logp; a.mean = mean; a.eps = eps;
    a.obs_dim = h->obs_dim; a.act_dim = h->act_dim; a.deterministic = deterministic ? 1 : 0; a.logp_const = h->logp_const;
    a.seed = seed; a.env_id0 = env_id0; a.step = step;
    a.log_std = log_std; a.noise = h->noise ? 1 : 0;
    for (int k = 0; k < NOUT; ++k) a.noise_std[k] = h->noise_std[k];
    const int64_t tiles = (n + TILE - 1) / TILE;
    const int64_t cap = 2 * (int64_t)h->sm_count;
    const unsigned grid = (unsigned)(tiles < cap ? tiles : cap);
    const bool squashed = h->head == HEAD_SQUASHED;
    if (h->mma_sync) {
        if (squashed) policy_act_kernel<HEAD_SQUASHED><<<grid, THREADS, PACKED_BYTES_SQUASHED, (cudaStream_t)stream>>>(a);
        else policy_act_kernel<HEAD_FIXED><<<grid, THREADS, PACKED_BYTES, (cudaStream_t)stream>>>(a);
    } else {
        a.packed = h->packed5;
        const int64_t cap5 = (tc5::GROUPS == 1 ? 2 : 1) * (int64_t)h->sm_count;   // small batches: one tile per SM before a second group gets one
        const unsigned grid5 = (unsigned)(tiles < cap5 ? tiles : cap5);
        if (squashed) tc5::policy_act_tc5_kernel<HEAD_SQUASHED><<<grid5, tc5::GT * tc5::GROUPS, tc5::SMEM_BYTES, (cudaStream_t)stream>>>(a);
        else tc5::policy_act_tc5_kernel<HEAD_FIXED><<<grid5, tc5::GT * tc5::GROUPS, tc5::SMEM_BYTES, (cudaStream_t)stream>>>(a);
    }
    return mvrl_check_launch("policy_act");
}

extern "C" MVRL_API int mvrl_policy_act(MvrlPolicy* h, int64_t n, int64_t ld, const float* obs, float* act, float* logp, float* mean,
                                        float* eps, uint64_t seed, uint64_t env_id0, uint32_t step, int deterministic, mvrl_stream_t stream) {
    return mvrl_policy_act_ex(h, n, ld, obs, act, logp, mean, nullptr, eps, seed, env_id0, step, deterministic, stream);
}
