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
//    the next after bias + GELU + bf16 packing.  The weights (70 KB as bf16, pre-packed in B-fragment order by policy_pack_kernel) sit
//    in shared memory; persistent grid, 2 CTAs per SM.  It re-reads every weight fragment for each 16 rows (587 MB of
//    shared-memory traffic per 131 072-env launch) and takes 42 us where the tcgen05 kernel takes 23; it stays as the
//    second implementation the tests compare the default against (same bf16 rounding, GELU code and Philox streams).
//  * policy_act_fp32_kernel (namespace f32, MVRL_POLICY_PRECISION_FP32): the network in fp32 as SB3 evaluates it - split-bf16
//    operands with three tcgen05.mma per K step, erf GELU, tanhf mean - for evaluating a trained agent.  Description above it.
//  * critic_target_kernel (namespace crit): SB3 SAC / TQC's critic target of a replay sample - the fp32 actor's next action,
//    n_critics critics streamed layer by layer from L2, TQC's sort / truncation or SAC's minimum.  Description above it.
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
// and the packing kernel halves the next layer's weights (a power of two: exact in bf16 and in the fp32 accumulation, so nothing changes
// numerically) - one packed multiply fewer per pair of columns
__device__ __forceinline__ unsigned gelu2x_pack2(float x0, float x1) {
    const float2 x = make_float2(x0, x1);
    const float2 x2 = __fmul2_rn(x, x);
    const float2 u = __fmul2_rn(x, __ffma2_rn(x2, make_float2(0.0356774081f, 0.0356774081f), make_float2(0.7978845608f, 0.7978845608f)));
    const float2 th = make_float2(tanh_fast(u.x), tanh_fast(u.y));
    const float2 y = __ffma2_rn(x, th, x);
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
// policy's eps, stream 8 the squashed head's action noise, stream 10 the critic target's eps and stream 11 the eps of the
// learner's action_log_prob (the counter words of 10 and 11 hold the sampled row and the 64-bit device call number where
// the actor's hold the env id and the step)
constexpr unsigned STREAM_EPS = 7u, STREAM_NOISE = 8u, STREAM_TARGET = 10u, STREAM_ACTOR_GRAD = 11u;
__device__ __forceinline__ float2 normal_pair(unsigned long long seed, unsigned long long env, unsigned step, unsigned blk,
                                              unsigned stream = STREAM_EPS) {
    const uint4 w = Philox::draw(seed, env, step, stream, blk);
    // [2^-25, 1], not (0, 1): the add rounds to even for k >= 2^23, so k = 2^24 - 1 gives u1 = 1 exactly (r = 0)
    const float u1 = (float(w.x >> 8) + 0.5f) * (1.0f / 16777216.0f);
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

// the draws of action pair pr (columns 2 pr, 2 pr + 1) of environment row r: eps and, for the squashed head with action
// noise, xi; zeros for a deterministic call and for a pair past act_dim
template <int HEAD>
__device__ __forceinline__ void draw_pair(const PolicyArgs& a, long r, int pr, float2& eps, float2& xi) {
    eps = xi = make_float2(0.0f, 0.0f);
    if (a.deterministic || 2 * pr >= a.act_dim) return;
    const unsigned long long env = a.env_id0 + (unsigned long long)r;
    eps = normal_pair(a.seed, env, a.step, (unsigned)pr);
    if (HEAD == HEAD_SQUASHED && a.noise) xi = normal_pair(a.seed, env, a.step, (unsigned)pr, STREAM_NOISE);
}

// the action head of environment row r for the pair (col, col + 1), col < act_dim, in all three kernels: h0, h1 = the first
// head layer's outputs (fixed: the mean's, squashed: mu's) and l0, l1 = the squashed head's log_std layer's, all without
// their biases (b4, sd).  Stores act / mean / log_std / eps when ok and returns the pair's log-prob terms.  ACCURATE: tanhf
// for the fixed head's mean (the fp32 kernel), else tanh.approx
template <int HEAD, bool ACCURATE>
__device__ __forceinline__ float head_pair(const PolicyArgs& a, const float* b4, const float* sd, int col, float h0, float h1,
                                           float l0, float l1, float2 e, float2 xi, long r, bool ok) {
    const bool second = col + 1 < a.act_dim;
    float m0, m1, o0, o1, s0 = 0.0f, s1 = 0.0f, lp;
    if constexpr (HEAD == HEAD_SQUASHED) {
        m0 = h0 + b4[col]; m1 = h1 + b4[col + 1];
        // noise_std is zero from act_dim on (set_squashed_noise)
        const Squashed q0 = squash(m0, l0 + sd[col], e.x, xi.x, a.noise_std[col]);
        const Squashed q1 = squash(m1, l1 + sd[col + 1], e.y, xi.y, a.noise_std[col + 1]);
        o0 = q0.act; o1 = q1.act; s0 = q0.ls; s1 = q1.ls;
        lp = q0.lp + (second ? q1.lp : 0.0f);
    } else {
        m0 = ACCURATE ? tanhf(h0 + b4[col]) : tanh_fast(h0 + b4[col]);
        m1 = ACCURATE ? tanhf(h1 + b4[col + 1]) : tanh_fast(h1 + b4[col + 1]);
        o0 = fminf(1.0f, fmaxf(-1.0f, fmaf(sd[col], e.x, m0)));
        o1 = fminf(1.0f, fmaxf(-1.0f, fmaf(sd[col + 1], e.y, m1)));
        lp = -0.5f * (e.x * e.x + (second ? e.y * e.y : 0.0f));
    }
    if (ok) {
        auto put = [&](float* dst, float v0, float v1) {   // dst: nullable
            if (!dst) return;
            dst[(long)col * a.ld + r] = v0;
            if (second) dst[(long)(col + 1) * a.ld + r] = v1;
        };
        a.act[(long)col * a.ld + r] = o0;
        if (second) a.act[(long)(col + 1) * a.ld + r] = o1;
        put(a.mean, m0, m1);
        if constexpr (HEAD == HEAD_SQUASHED) put(a.log_std, s0, s1);
        put(a.eps, e.x, e.y);
    }
    return lp;
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
            load_obs(tile + gridDim.x, a_next);
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
        float c5[4] = {0.0f, 0.0f, 0.0f, 0.0f};
        if constexpr (HEAD == HEAD_SQUASHED) {   // second n-tile: the log_std layer (b4 = b_mu, sd = b_log_std)
            const uint2* wls = reinterpret_cast<const uint2*>(smem + OFF_WLS);
#pragma unroll
            for (int kk = 0; kk < 8; ++kk) mma_bf16(c5, afr[kk], wls[kk * 32 + lane]);
        }
        if (col < a.act_dim) {
            // both rows' draws under one branch: draw_pair per row cost this kernel 8 instructions and 0.5 % (B200, 1000 W)
            float2 e0 = make_float2(0.0f, 0.0f), e1 = e0, x0 = e0, x1 = e0;
            if (!a.deterministic) {
                e0 = normal_pair(a.seed, a.env_id0 + (unsigned long long)r0, a.step, (unsigned)t);
                e1 = normal_pair(a.seed, a.env_id0 + (unsigned long long)r1, a.step, (unsigned)t);
                if (HEAD == HEAD_SQUASHED && a.noise) {
                    x0 = normal_pair(a.seed, a.env_id0 + (unsigned long long)r0, a.step, (unsigned)t, STREAM_NOISE);
                    x1 = normal_pair(a.seed, a.env_id0 + (unsigned long long)r1, a.step, (unsigned)t, STREAM_NOISE);
                }
            }
            lp0 = head_pair<HEAD, false>(a, b4, sd, col, c4[0], c4[1], c5[0], c5[1], e0, x0, r0, ok0);
            lp1 = head_pair<HEAD, false>(a, b4, sd, col, c4[2], c4[3], c5[2], c5[3], e1, x1, r1, ok1);
        }
        // log-prob: sum over the action columns = over the four lanes of a quad
        lp0 += __shfl_xor_sync(0xffffffffu, lp0, 1); lp0 += __shfl_xor_sync(0xffffffffu, lp0, 2);
        lp1 += __shfl_xor_sync(0xffffffffu, lp1, 1); lp1 += __shfl_xor_sync(0xffffffffu, lp1, 2);
        if (a.logp != nullptr && t == 0) {
            if (ok0) a.logp[r0] = lp0 + a.logp_const;
            if (ok1) a.logp[r1] = lp1 + a.logp_const;
        }
    }
}

// =====================================================================================================================
// tcgen05 building blocks of the three tensor-memory kernels (policy_act_tc5_kernel, policy_act_fp32_kernel,
// critic_target_kernel)
// =====================================================================================================================
constexpr int TM = 128;               // rows (environments, samples) per tile = TMEM lanes = threads per tile group
constexpr int A_BYTES = TM * H * 2;   // one tile's activations [128 x 128] bf16, canonical K-major

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
// the MMAs this thread has issued arrive on the mbarrier when they complete
__device__ __forceinline__ void mma_commit(unsigned bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tmem_ld16(unsigned taddr, unsigned (&v)[16]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]), "=r"(v[10]),
                   "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
                 : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tmem_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
// an mbarrier with one arrival per phase (a commit, or the expect_tx of a bulk load)
__device__ __forceinline__ void mbar_init(unsigned bar) { asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar)); }
__device__ __forceinline__ void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_wait(unsigned bar, unsigned parity) {
    unsigned done = 0;
    while (!done)
        asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2; selp.u32 %0, 1, 0, p; }"
                     : "=r"(done) : "r"(bar), "r"(parity) : "memory");
}
// the phase of bar completes when `bytes` have arrived through bulk copies (and the arrival of this call)
__device__ __forceinline__ void mbar_expect_tx(unsigned bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
// global -> shared memory at dst, bytes a multiple of 16; the bytes count towards the phase of bar
__device__ __forceinline__ void bulk_copy(void* dst, const void* src, unsigned bytes, unsigned bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"((unsigned)__cvta_generic_to_shared(dst)), "l"(src), "r"(bytes), "r"(bar) : "memory");
}
// the BYTES-byte parameter block, global -> shared memory at dst, as one bulk copy that completes the phase of bar
template <int BYTES>
__device__ __forceinline__ void load_params(void* dst, const void* src, unsigned bar) {
    mbar_expect_tx(bar, BYTES);
    bulk_copy(dst, src, BYTES, bar);
}
// on either side of a thread barrier: tcgen05 operations before it are ordered before tcgen05 operations after it
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
// COLS tensor-memory columns for the CTA, by warp 0, at the start of a kernel (after its mbarrier initialisation): every
// thread finds the base address in *slot after this
template <int COLS>
__device__ __forceinline__ void tmem_cta_alloc(unsigned* slot) {
    if (threadIdx.x < 32) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"((unsigned)__cvta_generic_to_shared(slot)), "n"(COLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
}
// ... and its release at the end, after every thread's last tcgen05 operation
template <int COLS>
__device__ __forceinline__ void tmem_cta_free(unsigned base) {
    tc_fence_before();
    __syncthreads();
    if (threadIdx.x < 32) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(base), "n"(COLS) : "memory");
}
// before the barrier that hands the A operand this thread has just stored (and the accumulator it has drained) to the
// MMA-issuing thread: its shared-memory stores are made visible to the tensor core's (async proxy) reads
__device__ __forceinline__ void fence_handoff() {
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    tc_fence_before();
}
// that hand-off in the single-group kernels (one tile group = the CTA)
__device__ __forceinline__ void publish() {
    fence_handoff();
    __syncthreads();
    tc_fence_after();
}
// this thread's accumulator row (128 columns from taddr) in 16-column chunks, double-buffered: the tcgen05.ld of chunk
// ch + 1 is in flight while chunk(w, c0) works on the columns c0 .. c0 + 15 of chunk ch (tcgen05.wait::ld waits for every
// outstanding load of the thread, so it comes AFTER that work)
template <class Chunk>
__device__ __forceinline__ void for_acc_chunks(unsigned taddr, Chunk chunk) {
    constexpr int NCH = H / 16;
    unsigned v[2][16];
    tmem_ld16(taddr, v[0]);
    tmem_wait_ld();
#pragma unroll
    for (int ch = 0; ch < NCH; ++ch) {
        if (ch + 1 < NCH) tmem_ld16(taddr + (unsigned)(16 * ch + 16), v[(ch + 1) & 1]);
        chunk(v[ch & 1], 16 * ch);
        if (ch + 1 < NCH) tmem_wait_ld();
    }
}

// the observation row of environment tile * TM + row (obs [obs_dim][ld]), zero-padded to K = 16; zeros for a tile past
// n_tiles or a row past n.  n_tiles and row by reference: so the tc5 kernel compiles to the SASS it was measured with (by
// value, the squashed instantiation's Philox XORs come out with their operands swapped)
__device__ __forceinline__ void load_obs(const PolicyArgs& a, const long& n_tiles, long tile, const int& row, float (&x)[KIN]) {
    const long r = tile * TM + row;
    const bool ok = tile < n_tiles && r < a.n;
#pragma unroll
    for (int k = 0; k < KIN; ++k) x[k] = (ok && k < a.obs_dim) ? a.obs[(long)k * a.ld + r] : 0.0f;
}

// the action head of row r once the head MMA has completed: this thread's 16 accumulator columns at tmem_row (the first
// head layer's outputs in 0..7, the squashed head's log_std layer's in 8..15) through head_pair, pair by pair below
// act_dim; b4 = the head biases b4[8] then std[8].  Returns the row's log-prob terms
template <int HEAD, bool ACCURATE>
__device__ __forceinline__ float head_row(const PolicyArgs& a, unsigned tmem_row, const float* b4, const float2 (&eps)[NOUT / 2],
                                          const float2 (&xi)[NOUT / 2], long r, bool ok) {
    unsigned hv[16];
    tmem_ld16(tmem_row, hv);
    tmem_wait_ld();
    const float* sd = b4 + NOUT;
    float lp = 0.0f;
#pragma unroll
    for (int pr = 0; pr < NOUT / 2; ++pr) {
        const int col = 2 * pr;
        if (col < a.act_dim)
            lp += head_pair<HEAD, ACCURATE>(a, b4, sd, col, __uint_as_float(hv[col]), __uint_as_float(hv[col + 1]),
                                            __uint_as_float(hv[NOUT + col]), __uint_as_float(hv[NOUT + col + 1]), eps[pr], xi[pr], r, ok);
    }
    return lp;
}

// ---- split-bf16 layers of the fp32 kernels (policy_act_fp32_kernel, critic_target_kernel): every operand x is stored as
// hi = bf16_rn(x) and lo = bf16_rn(x - hi), the A operand's lo A_BYTES after its hi, a weight matrix's lo w_bytes after its hi

// two fp32 values -> their bf16x2 hi and lo words: hi = bf16_rn(y), lo = bf16_rn(y - hi) (y - hi is exact in fp32)
__device__ __forceinline__ void split_pack2(float y0, float y1, unsigned& hi, unsigned& lo) {
    hi = pack_bf16(y0, y1);
    lo = pack_bf16(y0 - __uint_as_float(hi << 16), y1 - __uint_as_float(hi & 0xffff0000u));
}
// torch.nn.GELU(): x / 2 (1 + erf(x / sqrt 2)), fp32 with the accurate erff
__device__ __forceinline__ float gelu_erf(float x) {
    const float h = 0.5f * x;
    return fmaf(h, erff(x * 0.707106781186547524f), h);
}
// a K = 16 input row, split, as this thread's row of the A operands of a first layer (a_row16: its row in the K = 16 layout)
__device__ __forceinline__ void put_split_row16(unsigned char* a_row16, const float (&v)[KIN]) {
#pragma unroll
    for (int c = 0; c < KIN / 8; ++c) {
        unsigned hi[4], lo[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) split_pack2(v[8 * c + 2 * e], v[8 * c + 2 * e + 1], hi[e], lo[e]);
        *reinterpret_cast<uint4*>(a_row16 + c * 128) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
        *reinterpret_cast<uint4*>(a_row16 + A_BYTES + c * 128) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
    }
}
// hidden-layer epilogue: this thread's accumulator row (bias included) -> erf GELU in fp32 -> hi / lo bf16 -> its row of the
// next layer's A operands (a_row128: its row in the K = 128 layout)
__device__ __forceinline__ void gelu_split_row(unsigned tmem_row, unsigned char* a_row128) {
    for_acc_chunks(tmem_row, [&](const unsigned (&w)[16], int c0) {
#pragma unroll
        for (int q = 0; q < 2; ++q) {     // 8 columns = one 16-byte chunk of the row
            unsigned hi[4], lo[4];
#pragma unroll
            for (int e = 0; e < 4; ++e)
                split_pack2(gelu_erf(__uint_as_float(w[8 * q + 2 * e])), gelu_erf(__uint_as_float(w[8 * q + 2 * e + 1])), hi[e], lo[e]);
            *reinterpret_cast<uint4*>(a_row128 + ((c0 >> 3) + q) * 128) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
            *reinterpret_cast<uint4*>(a_row128 + A_BYTES + ((c0 >> 3) + q) * 128) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
        }
    });
}
// one layer, by one thread: D[128 x N] (+)= A[128 x K] B[N x K]^T into TMEM column d as three products per K = 16 step,
// A_hi B_hi + A_lo B_hi + A_hi B_lo (the dropped A_lo B_lo is 2^-16 relative); with `bias`, + 1 b^T: one more K = 16 step
// with A = the ones block and B = the bias as three bf16 terms (their sum is the fp32 bias); then commit -> bar
__device__ __forceinline__ void issue_split_layer(unsigned d, unsigned a_hi, unsigned a_lo, unsigned w, unsigned w_bytes, int K, int N,
                                                  bool bias, unsigned bias_addr, unsigned ones, unsigned bar) {
    const unsigned sbo = (unsigned)(K / 8) * 128u;
    const unsigned long long ah = smem_desc(a_hi, 128u, sbo), al = smem_desc(a_lo, 128u, sbo);
    const unsigned long long bh = smem_desc(w, 128u, sbo), bl = smem_desc(w + w_bytes, 128u, sbo);
    const unsigned idesc = instr_desc(TM, N);
    for (int j = 0; j < K / 16; ++j) {      // a K = 16 step is two 128-byte core-matrix columns: 256 bytes = 16 descriptor units
        const unsigned long long o = (unsigned long long)(16 * j);
        mma_ss(d, ah + o, bh + o, idesc, j > 0 ? 1u : 0u);
        mma_ss(d, al + o, bh + o, idesc, 1u);
        mma_ss(d, ah + o, bl + o, idesc, 1u);
    }
    if (bias) mma_ss(d, smem_desc(ones, 128u, 256u), smem_desc(bias_addr, 128u, 256u), idesc, 1u);
    mma_commit(bar);
}

// =====================================================================================================================
// tcgen05 version of the same network (the default).  A tile is 128 environments = the 128 lanes of tensor memory; a tile
// group of 128 threads (thread = one environment's row = one TMEM lane) takes one tile at a time through the network.  Per
// layer ONE thread of the group issues tcgen05.mma (M = 128, K = 16 per instruction, bf16 operands from shared memory through
// matrix descriptors, fp32 accumulator in the group's 128 TMEM columns) and commits to the group's mbarrier; the group's four
// warps then read their lane quadrant of the accumulator with tcgen05.ld, apply GELU, pack to bf16 and store the row into the
// A operand of the next layer - in the canonical K-major core-matrix layout (8 rows x 16 bytes contiguous; LBO = 128 B
// between the K-chunks, SBO = (K / 8) * 128 B between 8-row groups; no swizzle), so the store of 8 consecutive lanes is one
// contiguous 128-byte line.  Weights sit in shared memory in the same layout (packed by policy_pack_kernel), read by the
// tensor core ONCE per 128-row tile - the mma.sync version re-reads every B fragment for each 16 rows, 587 MB of
// shared-memory traffic per launch, its largest single cost.  The hidden biases are one more K = 16 MMA step per layer, so
// the epilogue reads and adds none (6 % faster than adding them there).
//
// ONE CTA per SM with GROUPS = 4 tile groups, which share only the weights and run out of phase: one group's MMA and
// barrier waits are filled by the others' epilogues (2 / 3 groups: 45 / 40 us against 32 us with 4).  Two threads per row
// (8 warps per tile, 64 columns each) measured slower: 34.0 vs 31.9 us, and 28.8 vs 24.4 us with the turn schedule of the
// kernel.  Same bf16 operand rounding, same GELU code, same Philox streams as the mma.sync kernel above (kept for A/B:
// MVRL_POLICY_MMA_SYNC=1); only the fp32 summation order inside the tensor core differs.
// =====================================================================================================================
namespace tc5 {

constexpr int HEAD_N = 16;                  // action columns padded to the smallest N of an M = 128 MMA
constexpr int OFF_W1 = 0;                     // [128 x 16]  bf16, canonical K-major
constexpr int OFF_W2 = OFF_W1 + H * KIN * 2;  // [128 x 128]
constexpr int OFF_W3 = OFF_W2 + H * H * 2;
constexpr int OFF_W4 = OFF_W3 + H * H * 2;    // [16 x 128]
constexpr int OFF_B = OFF_W4 + HEAD_N * H * 2;                  // float b1[128] b2[128] b3[128] b4[8] std[8]
constexpr int OFF_BIAS = OFF_B + (3 * H + 2 * NOUT) * 4;        // 3 x [128 x 16] bf16, canonical K-major: columns 0..2 = the bias split into three bf16 terms
constexpr int OFF_ONES = OFF_BIAS + 3 * H * KIN * 2;            // [128 x 16] bf16, canonical K-major: columns 0..2 = 1
constexpr int PARAM_BYTES = OFF_ONES + TM * KIN * 2;
constexpr int OFF_A = (PARAM_BYTES + 127) / 128 * 128;          // activations [128 x 128] bf16 per tile group, canonical K-major
constexpr int GROUPS = 4;                     // tile groups (= tiles in flight) per CTA; one CTA per SM
constexpr int SMEM_BYTES = OFF_A + GROUPS * A_BYTES;
constexpr int TMEM_COLS = GROUPS * H;         // the fp32 accumulator of one 128 x 128 layer per group (the head reuses its first 16)
static_assert(TMEM_COLS <= 512 && SMEM_BYTES <= 227 * 1024, "tile groups per CTA limited by TMEM columns and shared memory");
static_assert(PARAM_BYTES % 16 == 0, "parameter block is copied with 16-byte accesses");

template <int HEAD>
__global__ void __launch_bounds__(TM * GROUPS, 1) policy_act_tc5_kernel(const __grid_constant__ PolicyArgs a) {
    extern __shared__ __align__(128) unsigned char smem[];
    __shared__ __align__(8) unsigned long long mma_bars[GROUPS];
    __shared__ __align__(8) unsigned long long weights_bar;
    __shared__ unsigned tmem_base_slot;
    // a tile group owns one tile at a time: its own A operand buffer, accumulator columns, mbarrier and named barrier
    const int group = threadIdx.x / TM, row = threadIdx.x % TM;
    const unsigned bar = (unsigned)__cvta_generic_to_shared(&mma_bars[group]);
    const unsigned wbar = (unsigned)__cvta_generic_to_shared(&weights_bar);
    if (row == 0) {
        mbar_init(bar);
        if (group == 0) mbar_init(wbar);
        fence_mbar_init();
    }
    tmem_cta_alloc<TMEM_COLS>(&tmem_base_slot);
    // parameters: global (L2) -> shared, once per CTA, as ONE bulk copy (73 KB) that lands while the first observations are
    // fetched and packed; every thread waits for it once, before its group's first MMA / bias read.  (Copied by the threads
    // with 16-byte loads it was 14 % of the kernel's stall samples: nine dependent L2 round trips per thread.)
    if (threadIdx.x == 0) load_params<PARAM_BYTES>(smem, a.packed, wbar);
    const unsigned tmem_all = tmem_base_slot;
    const unsigned tmem_d = tmem_all + (unsigned)(group * H);
    const unsigned tmem_row = tmem_d + ((unsigned)(row & ~31) << 16);   // this warp's lane quadrant
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
        if (bias_off >= 0)   // + 1 b^T: one more K = 16 step, A = the constant ones block, B = the bias as three bf16 terms (their sum is the fp32 bias)
            mma_ss(tmem_d, smem_desc(smem_base + OFF_ONES, 128u, 256u), smem_desc(smem_base + bias_off, 128u, 256u), idesc, 1u);
        mma_commit(bar);
    };
    auto wait_layer = [&]() {
        mbar_wait(bar, parity);
        parity ^= 1u;
        tc_fence_after();
    };
    // hand the freshly written A operand (and the drained accumulator) over to the MMA-issuing thread
    auto publish_group = [&]() {
        fence_handoff();
        asm volatile("bar.sync %0, %1;" ::"r"(group + 1), "n"(TM) : "memory");   // this group only
        tc_fence_after();
    };
    // tiles are dealt out to the SMs first (tile t -> CTA t % gridDim.x), then to the groups of a CTA: every SM gets the same
    // number of tiles +- 1 (131 072 envs: 7 or 6 per SM; dealt to groups first, 108 SMs had 8 and 40 SMs had 4)
    const long n_tiles = (a.n + TM - 1) / TM;
    const long tile_step = (long)gridDim.x * GROUPS;
    const long first_tile = (long)blockIdx.x + (long)gridDim.x * group;
    float x[KIN];
    load_obs(a, n_tiles, first_tile, row, x);
    mbar_wait(wbar, 0u);   // the parameter block has landed (async proxy -> visible to the tensor core and, after this wait, to this thread)
    // PING-PONG.  Left alone, the four groups of a CTA run in lock step: they share the XU pipe fairly, so their epilogues
    // end together, their MMAs are issued together and queue on the one tensor core (each group then waits ~2000 cycles for
    // 576 cycles of MMA), and the XU pipe idles meanwhile - a third of a tile's 21.5 k cycles was MMA wait (clock64 trace,
    // tools/exp/actor_trace.py).  So the groups are split into two pairs that take turns: a pair enters a hidden-layer
    // epilogue only when the other pair has left its own (two named barriers, bar.sync by the pair that waits, bar.arrive by
    // the pair that leaves; all GROUPS * TM threads take part in a barrier phase) - while one pair keeps the XU pipe busy, the
    // other pair's MMAs run and complete.  Every group goes through the same number of turns; a group without a tile in an
    // iteration just passes the turn on.  (Also measured: single groups in round-robin order with at most 1 / 2 / 3 in the
    // epilogue at a time, by counters polled in shared memory: 29.6 / 24.8 / 25.3 us against 24.2 us for this pair scheme -
    // tools/exp/r2ab.sh.  Free-running groups: 26.5 us.  Named barriers cannot count: a group that runs two epilogues ahead of
    // its waiter completes a barrier phase on its own, and the CTA dead-locks.)
    const int pair = group >> 1;
    const long tiles_cta = (long)blockIdx.x < n_tiles ? (n_tiles - 1 - (long)blockIdx.x) / (long)gridDim.x + 1 : 0;   // tiles dealt to this CTA
    const long iters = (tiles_cta + GROUPS - 1) / GROUPS;
    long turn = 0;
    const long turns = 3 * iters;
    auto enter_epilogue = [&]() { asm volatile("bar.sync %0, %1;" ::"r"(5 + pair), "n"(GROUPS * TM) : "memory"); };
    auto leave_epilogue = [&]() {
        ++turn;
        if (!(pair == 1 && turn == turns)) asm volatile("bar.arrive %0, %1;" ::"r"(5 + (pair ^ 1)), "n"(GROUPS * TM) : "memory");
    };
    if (pair == 1 && turns > 0) asm volatile("bar.arrive %0, %1;" ::"r"(5), "n"(GROUPS * TM) : "memory");   // the first turn is pair 0's
    for (long it = 0; it < iters; ++it) {
        const long tile = first_tile + it * tile_step;
        if (tile >= n_tiles) {      // no tile for this group in this iteration: pass the three turns on
            for (int layer = 0; layer < 3; ++layer) { enter_epilogue(); leave_epilogue(); }
            continue;
        }
        const long r = tile * TM + row;
        const bool ok = r < a.n;
        // ---- this environment's observation row as the K = 16 A operand of layer 1
#pragma unroll
        for (int c = 0; c < KIN / 8; ++c)
            *reinterpret_cast<uint4*>(a_row16 + c * 128) = make_uint4(pack_bf16(x[8 * c], x[8 * c + 1]), pack_bf16(x[8 * c + 2], x[8 * c + 3]),
                                                                      pack_bf16(x[8 * c + 4], x[8 * c + 5]), pack_bf16(x[8 * c + 6], x[8 * c + 7]));
        publish_group();
        if (row == 0) issue_layer(OFF_W1, KIN, H, OFF_BIAS);
        load_obs(a, n_tiles, tile + tile_step, row, x);   // the next tile's observations travel while this tile runs through the network
        // the Gaussian noise of this environment's action pairs does not depend on the network: one Philox block + Box-Muller
        // per MMA in flight, computed in the shadow of the tensor core instead of after the head (29.2 -> 25.7 us)
        float2 eps[NOUT / 2], xi[NOUT / 2];   // xi: the squashed head's action noise
        draw_pair<HEAD>(a, r, 0, eps[0], xi[0]);
#pragma unroll
        for (int layer = 0; layer < 3; ++layer) {
            wait_layer();
            enter_epilogue();
            // ---- epilogue of hidden layer `layer`: accumulator row (bias included) -> GELU -> bf16 -> A operand of the next
            // layer.  With the turn schedule only two warps per scheduler are in an epilogue and nothing else hides the TMEM
            // read latency, hence the double-buffered read (24.05 -> 22.85 us; free-running groups: 26.1 vs 25.7 us)
            for_acc_chunks(tmem_row, [&](const unsigned (&w)[16], int c0) {
#pragma unroll
                for (int q = 0; q < 2; ++q) {     // 8 columns = one 16-byte chunk of the row
                    unsigned pk[4];
#pragma unroll
                    for (int e = 0; e < 4; ++e) pk[e] = gelu2x_pack2(__uint_as_float(w[8 * q + 2 * e]), __uint_as_float(w[8 * q + 2 * e + 1]));
                    *reinterpret_cast<uint4*>(a_row128 + ((c0 >> 3) + q) * 128) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
                }
            });
            leave_epilogue();
            publish_group();
            if (row == 0) {
                if (layer < 2) issue_layer(layer == 0 ? OFF_W2 : OFF_W3, H, H, OFF_BIAS + (layer + 1) * H * KIN * 2);
                else issue_layer(OFF_W4, H, HEAD_N, -1);     // the head biases are added in fp32 by head_pair
            }
            draw_pair<HEAD>(a, r, layer + 1, eps[layer + 1], xi[layer + 1]);
        }
        // ---- head: the action columns of this environment's row (squashed head: mu in accumulator columns 0..7, the log_std
        // layer in 8..15; b4 = b_mu, sd = b_log_std), Gaussian sample, log-prob
        wait_layer();
        const float lp = head_row<HEAD, false>(a, tmem_row, bias + 3 * H, eps, xi, r, ok);
        if (a.logp != nullptr && ok) a.logp[r] = lp + a.logp_const;
        // the next tile's first publish_group() orders these accumulator reads before the next layer-1 MMA overwrites TMEM
    }
    tmem_cta_free<TMEM_COLS>(tmem_all);
}

}  // namespace tc5

// =====================================================================================================================
// fp32-accurate version (MVRL_POLICY_PRECISION_FP32): the network SB3 evaluates - fp32 operands, GELU in its erf form
// (torch.nn.GELU()), the fixed head's mean with the accurate tanhf - on the same tcgen05 tensor core.  Every operand x is
// split into hi = bf16_rn(x) and lo = bf16_rn(x - hi) (16 significant bits together; bf16 has fp32's exponent range, so lo
// does not underflow as an fp16 split would), and every K = 16 step is three kind::f16 MMAs into the same fp32 TMEM
// accumulator: A_hi B_hi + A_lo B_hi + A_hi B_lo (the dropped A_lo B_lo is 2^-16 relative).  This applies to the
// observations, the hidden activations and the weights of all four layers; the hidden biases go through the fast kernel's
// three-term bias MMA (exact), the head biases are added in fp32 by the epilogue.
//
// Shared memory: the split doubles every operand - parameters 161.6 KB (W1 8 KB, W2 + W3 128 KB, head 8 KB, fp32 biases,
// bias-MMA blocks and ones 17.6 KB) + one tile's activations hi + lo (64 KB) = 225.6 KB of the 227 KB of a block.  So ONE
// tile group (128 threads, thread = one environment's row = one TMEM lane) per CTA and one CTA per SM: the activations are
// the A operand in shared memory as in the fast kernel, but there is no second tile whose epilogue would overlap this
// tile's MMAs.  The sampling, clamp and log-prob code and the Philox streams are the fast kernel's.
// =====================================================================================================================
namespace f32 {

constexpr int HEAD_N = tc5::HEAD_N;
constexpr int W1_BYTES = H * KIN * 2, WH_BYTES = H * H * 2, W4_BYTES = HEAD_N * H * 2;
constexpr int OFF_W1 = 0;                         // hi, then lo at + W1_BYTES: [128 x 16] bf16, canonical K-major
constexpr int OFF_W2 = OFF_W1 + 2 * W1_BYTES;     // hi, lo: [128 x 128]
constexpr int OFF_W3 = OFF_W2 + 2 * WH_BYTES;
constexpr int OFF_W4 = OFF_W3 + 2 * WH_BYTES;     // hi, lo: [16 x 128], the squashed head's log_std layer in rows 8..
constexpr int OFF_B = OFF_W4 + 2 * W4_BYTES;      // float b1[128] b2[128] b3[128] b4[8] std[8]
constexpr int OFF_BIAS = OFF_B + (3 * H + 2 * NOUT) * 4;   // 3 x [128 x 16]: the bias as three bf16 terms (tc5's bias MMA)
constexpr int OFF_ONES = OFF_BIAS + 3 * H * KIN * 2;
constexpr int PARAM_BYTES = OFF_ONES + TM * KIN * 2;
constexpr int OFF_A = (PARAM_BYTES + 127) / 128 * 128;    // activations hi, then lo: [128 x 128] bf16 each
constexpr int SMEM_BYTES = OFF_A + 2 * A_BYTES;
static_assert(PARAM_BYTES % 16 == 0, "parameter block is copied with 16-byte accesses");
static_assert(SMEM_BYTES + 64 <= 227 * 1024, "parameters + one tile's split activations + static shared memory");

template <int HEAD>
__global__ void __launch_bounds__(TM, 1) policy_act_fp32_kernel(const __grid_constant__ PolicyArgs a) {
    extern __shared__ __align__(128) unsigned char smem[];
    __shared__ __align__(8) unsigned long long mma_bar;
    __shared__ __align__(8) unsigned long long weights_bar;
    __shared__ unsigned tmem_base_slot;
    const int row = threadIdx.x;
    const unsigned bar = (unsigned)__cvta_generic_to_shared(&mma_bar);
    const unsigned wbar = (unsigned)__cvta_generic_to_shared(&weights_bar);
    if (row == 0) {
        mbar_init(bar);
        mbar_init(wbar);
        fence_mbar_init();
    }
    tmem_cta_alloc<H>(&tmem_base_slot);   // the fp32 accumulator of one 128 x 128 layer (the head uses the first 16)
    if (row == 0) load_params<PARAM_BYTES>(smem, a.packed, wbar);   // 162 KB, landing while the first observations are fetched
    const unsigned tmem_d = tmem_base_slot;
    const unsigned tmem_row = tmem_d + ((unsigned)(row & ~31) << 16);   // this warp's lane quadrant
    const unsigned smem_base = (unsigned)__cvta_generic_to_shared(smem);
    const unsigned a_hi = smem_base + OFF_A, a_lo = a_hi + A_BYTES;
    const float* bias = reinterpret_cast<const float*>(smem + OFF_B);
    unsigned char* a_row16 = smem + OFF_A + (row >> 3) * (KIN / 8 * 128) + (row & 7) * 16;   // this thread's row, K = 16 layout
    unsigned char* a_row128 = smem + OFF_A + (row >> 3) * (H / 8 * 128) + (row & 7) * 16;    // K = 128 layout
    auto issue_layer = [&](int w_off, int w_bytes, int K, int N, int bias_off) {
        issue_split_layer(tmem_d, a_hi, a_lo, smem_base + w_off, w_bytes, K, N, bias_off >= 0, smem_base + bias_off, smem_base + OFF_ONES, bar);
    };
    unsigned parity = 0;
    auto wait_layer = [&]() {
        mbar_wait(bar, parity);
        parity ^= 1u;
        tc_fence_after();
    };
    const long n_tiles = (a.n + TM - 1) / TM;
    float x[KIN];
    load_obs(a, n_tiles, blockIdx.x, row, x);
    mbar_wait(wbar, 0u);
    for (long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const long r = tile * TM + row;
        const bool ok = r < a.n;
        put_split_row16(a_row16, x);              // this environment's observation row: the A operands of layer 1
        publish();
        if (row == 0) issue_layer(OFF_W1, W1_BYTES, KIN, H, OFF_BIAS);
        load_obs(a, n_tiles, tile + gridDim.x, row, x);   // the next tile's observations travel while this tile runs through the network
        float2 eps[NOUT / 2], xi[NOUT / 2];       // the noise does not depend on the network: drawn in the shadow of the layer-1 MMAs
#pragma unroll
        for (int pr = 0; pr < NOUT / 2; ++pr) draw_pair<HEAD>(a, r, pr, eps[pr], xi[pr]);
#pragma unroll 1
        for (int layer = 0; layer < 3; ++layer) {
            wait_layer();
            gelu_split_row(tmem_row, a_row128);
            publish();
            if (row == 0) {
                if (layer < 2) issue_layer(layer == 0 ? OFF_W2 : OFF_W3, WH_BYTES, H, H, OFF_BIAS + (layer + 1) * H * KIN * 2);
                else issue_layer(OFF_W4, W4_BYTES, H, HEAD_N, -1);   // the head biases are added in fp32 by head_pair
            }
        }
        // ---- head: as the fast kernel's, with tanhf for the fixed head's mean
        wait_layer();
        const float lp = head_row<HEAD, true>(a, tmem_row, bias + 3 * H, eps, xi, r, ok);
        if (a.logp != nullptr && ok) a.logp[r] = lp + a.logp_const;
        // the next tile's first publish() orders these accumulator reads before the next layer-1 MMA overwrites TMEM
    }
    tmem_cta_free<H>(tmem_d);
}

}  // namespace f32

// =====================================================================================================================
// Critic target of SB3 SAC / sb3_contrib TQC (K10): for a sampled batch, next action and log-prob by the fp32 squashed
// actor, n_critics critic MLPs on [next_obs, next_action], then the TQC truncated quantiles (sort, keep the smallest
// n_target) or SAC's minimum, and r + (1 - d) gamma (q - alpha logp) - in fp32 as SB3 computes it, with the fp32 actor's
// code: split-bf16 layers (put_split_row16, issue_split_layer, gelu_split_row) and its head (head_row).
//
// One CTA = one tile of 128 sampled rows, one row per thread and TMEM lane.  The weights of 1 + n_critics networks do not fit
// in shared memory (one fp32 network's hi / lo block is ~160 KB), so they are STREAMED layer by layer from L2 into a ring of
// two slots, each filled by bulk copies that complete the phase of the slot's mbarrier: the copy of layer g + 2 starts as soon
// as the MMAs of layer g (which read the same slot) have completed, so it lands while layer g + 1 multiplies.  A slot holds a
// layer's weights hi, lo and its bias as three bf16 terms (the bias MMA against a ones block, as in the fp32 actor): the
// largest, a hidden 128 x 128 layer, is 68 KB.  The layer sequence is the actor's four (read from the actor handle's packed
// block, unchanged) then four per critic (the critic layout below, packed by policy_pack_kernel).  TMEM: columns 0..127 are
// the hidden accumulator (the actor's head uses 0..15); critic c writes its n_quantiles outputs (N = nqp, n_quantiles rounded
// up to 16) to columns 128 + c nqp, where they stay until the last critic is done.  At the end of the tile the two slots are
// free and hold each row's n_critics n_quantiles values for a rank-based selection (count of smaller values, ties broken by
// index), which writes each kept value's label at its rank: the output row is sorted ascending.
// =====================================================================================================================
namespace crit {

constexpr int MAX_CRITICS = 5, MAX_QUANTILES = 32;
constexpr int BIAS_BYTES = H * KIN * 2;                          // the bias terms of a 128-wide layer: [128 x 16] bf16
// the packed block of one critic: per layer hi, lo (canonical K-major) then the bias terms ([N x 16], columns 0..2)
constexpr int L1_BYTES = 2 * f32::W1_BYTES + BIAS_BYTES;         // 12 KB
constexpr int LH_BYTES = 2 * f32::WH_BYTES + BIAS_BYTES;         // 68 KB
__host__ __device__ constexpr int out_bytes(int nqp) { return 2 * nqp * H * 2 + nqp * KIN * 2; }
__host__ __device__ constexpr int critic_bytes(int nqp) { return L1_BYTES + 2 * LH_BYTES + out_bytes(nqp); }
constexpr int SLOT_BYTES = LH_BYTES;                             // the largest layer
constexpr int OFF_A = 2 * SLOT_BYTES;                            // activations hi, then lo: [128 x 128] bf16 each
constexpr int OFF_ONES = OFF_A + 2 * A_BYTES;                    // [128 x 16] bf16, columns 0..2 = 1 (the bias MMA's A)
constexpr int OFF_ACT = OFF_ONES + TM * KIN * 2;                 // float [8][128]: head_pair's action output
constexpr int SMEM_BYTES = OFF_ACT + NOUT * TM * 4;
constexpr int SORT_LD = MAX_CRITICS * MAX_QUANTILES + 1;         // odd: thread t's value j is in bank (t + j) mod 32
constexpr int TMEM_COLS = 512;
static_assert(SMEM_BYTES + 64 <= 227 * 1024, "two slots + one tile's split activations + static shared memory");
static_assert(TM * SORT_LD * 4 <= OFF_A, "the sort rows overlay the two weight slots");
static_assert(H + MAX_CRITICS * MAX_QUANTILES <= TMEM_COLS, "hidden accumulator + every critic's outputs");
static_assert(SLOT_BYTES % 16 == 0 && L1_BYTES % 16 == 0 && out_bytes(16) % 16 == 0, "bulk copies move 16-byte units");

struct CriticArgs {
    const unsigned char* actor;    // the fp32 squashed actor's packed block (f32 layout)
    const unsigned char* critic;   // n_critics blocks of critic_bytes(nqp)
    long n;
    const float *next_obs, *rewards, *dones, *ent_coef;   // [n, obs_dim], [n], [n], [1]
    float gamma, logp_const;
    int obs_dim, act_dim, nc, nq, nqp, n_target;
    unsigned long long seed;
    long long* calls;              // [0] = calls, [1] = blocks arrived (0 between launches)
    float *target, *next_actions, *next_logp, *eps;         // [n, n_target]; nullable [n, act_dim], [n], [n, act_dim]
};

// where layer g of the sequence comes from and how it multiplies
struct Layer {
    const unsigned char *src0, *src1;   // bulk copies into the slot at 0 and at bytes0 (src1 nullable)
    int bytes0, bytes1, w_bytes, K, N, col;
    bool bias;
};
__device__ __forceinline__ Layer layer_of(const CriticArgs& a, int g) {
    Layer L;
    L.src1 = nullptr; L.bytes1 = 0; L.col = 0; L.bias = true; L.K = H; L.N = H;
    if (g < 4) {   // the actor: its weights hi / lo, then its bias terms (a separate region of its block)
        L.w_bytes = g == 0 ? f32::W1_BYTES : g < 3 ? f32::WH_BYTES : f32::W4_BYTES;
        L.src0 = a.actor + (g == 0 ? f32::OFF_W1 : g == 1 ? f32::OFF_W2 : g == 2 ? f32::OFF_W3 : f32::OFF_W4);
        L.bytes0 = 2 * L.w_bytes;
        if (g == 0) L.K = KIN;
        if (g < 3) { L.src1 = a.actor + f32::OFF_BIAS + g * BIAS_BYTES; L.bytes1 = BIAS_BYTES; }
        else { L.N = f32::HEAD_N; L.bias = false; }   // the head biases are added in fp32 by head_pair
        return L;
    }
    const int c = (g - 4) >> 2, l = (g - 4) & 3;
    const unsigned char* base = a.critic + (long)c * critic_bytes(a.nqp);
    if (l == 0) { L.src0 = base; L.bytes0 = L1_BYTES; L.w_bytes = f32::W1_BYTES; L.K = KIN; }
    else if (l < 3) { L.src0 = base + L1_BYTES + (l - 1) * LH_BYTES; L.bytes0 = LH_BYTES; L.w_bytes = f32::WH_BYTES; }
    else { L.src0 = base + L1_BYTES + 2 * LH_BYTES; L.bytes0 = out_bytes(a.nqp); L.w_bytes = a.nqp * H * 2; L.N = a.nqp; L.col = H + c * a.nqp; }
    return L;
}

__global__ void __launch_bounds__(TM, 1) critic_target_kernel(const __grid_constant__ CriticArgs a) {
    extern __shared__ __align__(128) unsigned char smem[];
    __shared__ __align__(8) unsigned long long mma_bar, slot_bars[2];
    __shared__ unsigned tmem_base_slot;
    __shared__ unsigned long long s_call;
    const int row = threadIdx.x;
    const unsigned bar = (unsigned)__cvta_generic_to_shared(&mma_bar);
    const unsigned sbar0 = (unsigned)__cvta_generic_to_shared(&slot_bars[0]), sbar1 = (unsigned)__cvta_generic_to_shared(&slot_bars[1]);
    auto slot_bar = [&](int g) { return (g & 1) ? sbar1 : sbar0; };
    if (row == 0) {
        mbar_init(bar);
        mbar_init(sbar0);
        mbar_init(sbar1);
        fence_mbar_init();
        s_call = device_call_number(&a.calls[0], &a.calls[1]);
    }
    tmem_cta_alloc<TMEM_COLS>(&tmem_base_slot);
    const int n_layers = 4 + 4 * a.nc;
    auto load_layer = [&](int g) {   // thread 0: layer g -> slot g % 2
        const Layer L = layer_of(a, g);
        unsigned char* dst = smem + (g & 1) * SLOT_BYTES;
        mbar_expect_tx(slot_bar(g), (unsigned)(L.bytes0 + L.bytes1));
        bulk_copy(dst, L.src0, (unsigned)L.bytes0, slot_bar(g));
        if (L.src1) bulk_copy(dst + L.bytes0, L.src1, (unsigned)L.bytes1, slot_bar(g));
    };
    if (row == 0) { load_layer(0); load_layer(1); }
    const unsigned tmem_d = tmem_base_slot;
    const unsigned tmem_row = tmem_d + ((unsigned)(row & ~31) << 16);   // this warp's lane quadrant
    const unsigned smem_base = (unsigned)__cvta_generic_to_shared(smem);
    const unsigned a_hi = smem_base + OFF_A, a_lo = a_hi + A_BYTES;
    unsigned char* a_row16 = smem + OFF_A + (row >> 3) * (KIN / 8 * 128) + (row & 7) * 16;   // this thread's row, K = 16 layout
    unsigned char* a_row128 = smem + OFF_A + (row >> 3) * (H / 8 * 128) + (row & 7) * 16;    // K = 128 layout
    // the ones block of the bias MMA, row by row (bias_mma_word's: columns 0..2 = bf16 1)
    *reinterpret_cast<uint4*>(smem + OFF_ONES + (row >> 3) * 256 + (row & 7) * 16) = make_uint4(0x3f803f80u, 0x3f80u, 0u, 0u);
    *reinterpret_cast<uint4*>(smem + OFF_ONES + (row >> 3) * 256 + (row & 7) * 16 + 128) = make_uint4(0u, 0u, 0u, 0u);
    // this row's sample
    const long r = (long)blockIdx.x * TM + row;
    const bool ok = r < a.n;
    float x[KIN];
#pragma unroll
    for (int k = 0; k < KIN; ++k) x[k] = (ok && k < a.obs_dim) ? a.next_obs[r * a.obs_dim + k] : 0.0f;
    const float rew = ok ? a.rewards[r] : 0.0f, done = ok ? a.dones[r] : 0.0f;
    put_split_row16(a_row16, x);
    // eps: stream 10, counter (row, call lo, call hi, 10 * 65536 + pair), key seed - normal_pair with the row and the call's
    // low word in the env id's two words and the call's high word in the step's; drawn while the first layers load
    float2 eps[NOUT / 2];
    const unsigned long long call = s_call;
#pragma unroll
    for (int pr = 0; pr < NOUT / 2; ++pr)
        eps[pr] = (ok && 2 * pr < a.act_dim)
                      ? normal_pair(a.seed, (unsigned long long)(unsigned)r | (call << 32), (unsigned)(call >> 32), (unsigned)pr, STREAM_TARGET)
                      : make_float2(0.0f, 0.0f);
    // head_pair's view: actions into shared memory (this thread's column r = row of [8][128]), no noise, nothing else written
    float* s_act = reinterpret_cast<float*>(smem + OFF_ACT);
    PolicyArgs pa{};
    pa.act = s_act; pa.ld = TM; pa.act_dim = a.act_dim;
    float lp = 0.0f;
    unsigned parity = 0;
#pragma unroll 1
    for (int g = 0; g < n_layers; ++g) {
        publish();
        if (row == 0) {
            const Layer L = layer_of(a, g);
            mbar_wait(slot_bar(g), (unsigned)(g >> 1) & 1u);
            const unsigned slot = smem_base + (unsigned)((g & 1) * SLOT_BYTES);
            issue_split_layer(tmem_d + (unsigned)L.col, a_hi, a_lo, slot, (unsigned)L.w_bytes, L.K, L.N, L.bias, slot + 2 * L.w_bytes,
                              smem_base + OFF_ONES, bar);
        }
        mbar_wait(bar, parity);
        parity ^= 1u;
        tc_fence_after();
        if (row == 0 && g + 2 < n_layers) load_layer(g + 2);   // the slot's MMAs are complete: refill it
        const int l = g & 3;
        if (l < 3) {   // hidden
            gelu_split_row(tmem_row, a_row128);
        } else if (g == 3) {   // the actor's head: mu in columns 0..7, log_std in 8..15 -> a, logp; the critics' input [obs, a]
            const float2 no_noise[NOUT / 2] = {};
            lp = head_row<HEAD_SQUASHED, true>(pa, tmem_row, reinterpret_cast<const float*>(a.actor + f32::OFF_B) + 3 * H, eps, no_noise, row, true);
            lp += a.logp_const;
#pragma unroll
            for (int k = 0; k < NOUT; ++k)
                if (k < a.act_dim) {
                    if (ok && a.next_actions) a.next_actions[r * a.act_dim + k] = s_act[k * TM + row];
                    if (ok && a.eps) a.eps[r * a.act_dim + k] = k & 1 ? eps[k >> 1].y : eps[k >> 1].x;
                }
            if (ok && a.next_logp) a.next_logp[r] = lp;
#pragma unroll
            for (int j = 0; j < KIN; ++j)   // the action columns follow the observation's (th.cat([obs, a], 1)); a select, not an indexed store
                if (j >= a.obs_dim && j < a.obs_dim + a.act_dim) x[j] = s_act[(j - a.obs_dim) * TM + row];
            put_split_row16(a_row16, x);
        } else if (g + 1 < n_layers) {   // a critic's output layer: its values stay in TMEM; the next critic's input
            put_split_row16(a_row16, x);
        }
    }
    // ---- every critic's outputs -> the kept values, r + (1 - d) gamma (q - alpha logp) in SB3's fp32 operation order
    const float alpha = *a.ent_coef, scale = __fmul_rn(1.0f - done, a.gamma);
    auto label = [&](float q) { return __fadd_rn(rew, __fmul_rn(scale, __fsub_rn(q, __fmul_rn(alpha, lp)))); };
    float* sort_row = reinterpret_cast<float*>(smem) + row * SORT_LD;   // the slots are free: every MMA has completed
    float qmin = INFINITY;
#pragma unroll 1
    for (int c = 0; c < a.nc; ++c)
#pragma unroll 1
        for (int h = 0; h < a.nqp; h += 16) {
            unsigned v[16];
            tmem_ld16(tmem_row + (unsigned)(H + c * a.nqp + h), v);
            tmem_wait_ld();
#pragma unroll
            for (int e = 0; e < 16; ++e)
                if (h + e < a.nq) {
                    qmin = fminf(qmin, __uint_as_float(v[e]));
                    sort_row[c * a.nq + h + e] = __uint_as_float(v[e]);
                }
        }
    if (a.n_target == 1) {   // SAC (min over the critics), or TQC keeping one value
        if (ok) a.target[r] = label(qmin);
    } else {   // rank of value i = #{j: v_j < v_i} + #{j < i: v_j == v_i}, 16 values at a time against every j
        const int n = a.nc * a.nq;
#pragma unroll 1
        for (int i0 = 0; i0 < n; i0 += 16) {
            float vi[16];
            int rk[16];
#pragma unroll
            for (int u = 0; u < 16; ++u) { vi[u] = i0 + u < n ? sort_row[i0 + u] : INFINITY; rk[u] = 0; }
#pragma unroll 4
            for (int j = 0; j < i0; ++j) {
                const float v = sort_row[j];
#pragma unroll
                for (int u = 0; u < 16; ++u) rk[u] += v <= vi[u] ? 1 : 0;
            }
#pragma unroll
            for (int j = 0; j < 16; ++j)
#pragma unroll
                for (int u = 0; u < 16; ++u)
                    if (j != u) rk[u] += (j < u ? vi[j] <= vi[u] : vi[j] < vi[u]) ? 1 : 0;
#pragma unroll 4
            for (int j = i0 + 16; j < n; ++j) {
                const float v = sort_row[j];
#pragma unroll
                for (int u = 0; u < 16; ++u) rk[u] += v < vi[u] ? 1 : 0;
            }
#pragma unroll
            for (int u = 0; u < 16; ++u)
                if (ok && i0 + u < n && rk[u] < a.n_target) a.target[r * a.n_target + rk[u]] = label(vi[u]);
        }
    }
    tmem_cta_free<TMEM_COLS>(tmem_d);
}

}  // namespace crit

// =====================================================================================================================
// The critics with gradients (K12): SB3's critic forward on [obs, act] and its backward pass to the parameters and the
// actions, in fp32 with the split-bf16 products of the critic target (the same packed block, packed by policy_pack_kernel).
//
// critic_forward_kernel: one CTA per 128-row tile and critic, one row per thread and TMEM lane, the critic's four layers
// streamed through crit's two slots (layer_of) and multiplied by issue_split_layer with the bias MMA; gelu_split_row is the
// epilogue.  With `saved`, the pre-activations z1..z3 are also stored in fp32, feature-major inside a tile
// ([critic][layer][tile][feature][row]), so that a warp's loads of one feature in the backward pass are 128 contiguous bytes.
//
// critic_backward_kernel: a CTA holds ONE critic and a fixed run of consecutive tiles (tiles_per_cta depends on B and
// n_critics only).  Per tile, from the output layer down:
//   dgrad  dH_{l-1} = dZ_l W_l into the layer accumulator, then dZ_{l-1} = dH_{l-1} GELU'(z_{l-1}) (torch's cdf + z pdf);
//          the packed W (canonical K-major [out][in]) is the B operand read MN-major: its 16-byte chunks are 8 input features
//          of one output row in both readings, so the transpose bit of the instruction descriptor turns W into W^T.
//   wgrad  dW_l += dZ_l^T H_{l-1} with K = the tile's 128 rows: both operands are the tiles the epilogue writes row by row
//          (split dZ, split H = gelu(z) recomputed from the saved z), read MN-major; the hidden biases are one more N = 16
//          product against the ones block; the output layer is accumulated transposed (H3^T dZ4, N = nqp) and its bias
//          is summed per thread in registers.
// The weight gradients stay in TMEM across the CTA's tiles; at the end each CTA writes one partial of every parameter to
// scratch and critic_grad_reduce_kernel adds the partials (and the critics' action gradients) in a fixed order.
//
// The actor with gradients (K13): the same three kernels instantiated with NET_ACTOR run SB3's Actor.action_log_prob and
// its backward pass to the actor's parameters.  Two pieces differ from the critics': the weight source (the fp32 squashed
// actor's packed block, f32 layout, walked by crit::layer_of for g < 4; layer 1's input is obs alone) and the output
// layer.  Forward: the squashed head's 16 accumulator columns (mu in 0..7, log_std in 8..15) go through head_row with eps
// from Philox stream 11, and with `saved` each row's mu, log_std pre-activation and eps are stored after z1..z3.
// Backward: dZ_head = [g_mu | g_ls] of each row from grad_actions, grad_log_prob and those saved values (actor_head_dz),
// then K12's dgrad / wgrad down to W1, without an input gradient.
// =====================================================================================================================
namespace cgrad {

using crit::MAX_CRITICS;
constexpr int NET_CRITIC = 0, NET_ACTOR = 1;            // which network the kernels below run
constexpr int BWD_CTAS = 144;                          // CTAs per launch at most, over all critics (one wave of a B200)
// TMEM columns of the backward kernel: the layer accumulator, then the weight-gradient accumulators of one network
constexpr int T_ACC = 0, T_W1 = 128, T_B1 = T_W1 + KIN, T_W2 = T_B1 + 16, T_B2 = T_W2 + H, T_W3 = T_B2 + 16, T_B3 = T_W3 + H,
              T_W4 = T_B3 + 16, T_END = T_W4 + crit::MAX_QUANTILES;
constexpr int BWD_TMEM_COLS = 512;
static_assert(T_END <= BWD_TMEM_COLS, "layer accumulator + dW1, db1, dW2, db2, dW3, db3, dW4^T of one critic");
static_assert(T_W4 + f32::HEAD_N <= BWD_TMEM_COLS, "layer accumulator + dW1 .. db3 and the squashed head's dW^T of the actor");
// the actor's saved values: z1..z3 as one critic's, then per tile [3 NOUT][TM] - mu, the log_std pre-activation (before the
// clamp) and eps of each action column, feature-major like z
__host__ __device__ constexpr long head_saved_offset(long n_tiles) { return 3 * n_tiles * (long)(H * TM); }
__host__ __device__ constexpr long actor_saved_floats(long n_tiles) { return head_saved_offset(n_tiles) + n_tiles * 3 * NOUT * TM; }
// shared memory of the backward kernel: one weight slot (hi, lo of the largest layer), split dZ and H tiles, the ones block
constexpr int B_OFF_W = 0, B_OFF_DZ = 2 * f32::WH_BYTES, B_OFF_H = B_OFF_DZ + 2 * A_BYTES, B_OFF_ONES = B_OFF_H + 2 * A_BYTES;
constexpr int BWD_SMEM_BYTES = B_OFF_ONES + TM * KIN * 2;
static_assert(BWD_SMEM_BYTES + 64 <= 227 * 1024, "weight slot + split dZ and H tiles + ones block + static shared memory");
static_assert(TM * (crit::MAX_QUANTILES + 1) * 4 <= 2 * A_BYTES, "the output bias sums overlay the H tile");
constexpr int FWD_SMEM_BYTES = crit::OFF_ONES + TM * KIN * 2;
// one CTA's partial: TMEM columns T_W1 .. T_W4 + nqp, lane-major ([column][lane]), then the output bias [MAX_QUANTILES]
__host__ __device__ constexpr long part_floats(int nqp) { return (long)(T_W4 - T_W1 + nqp) * TM + crit::MAX_QUANTILES; }
__host__ __device__ constexpr long tiles_per_cta(long n_tiles, int nc) {
    const long g = BWD_CTAS / nc;
    return (n_tiles + g - 1) / g;
}

struct FwdArgs {
    const unsigned char* net;          // the critics' blocks (crit layout) or the fp32 squashed actor's (f32 layout)
    long n, n_tiles;
    const float *obs, *act;
    float *q, *saved;
    int obs_dim, act_dim, nc, nq, nqp;
    // the actor: actions [n][act_dim], log_prob [n], eps [n][act_dim] (nullable); eps from stream 11 keyed on seed, row and
    // the device call number calls[0] (calls[1]: device_call_number's ticket)
    float *actions, *logp, *eps;
    unsigned long long seed;
    long long* calls;
    float logp_const;
};

// this thread's row of the critics' input [obs, act], zero-padded to K = 16 (zeros past n)
__device__ __forceinline__ void load_obs_act(const float* obs, const float* act, int obs_dim, int act_dim, long r, bool ok, float (&x)[KIN]) {
#pragma unroll
    for (int k = 0; k < KIN; ++k)
        x[k] = !ok ? 0.0f : k < obs_dim ? obs[r * obs_dim + k] : k < obs_dim + act_dim ? act[r * act_dim + (k - obs_dim)] : 0.0f;
}

template <int NET>
__global__ void __launch_bounds__(TM, 1) critic_forward_kernel(const __grid_constant__ FwdArgs a) {
    constexpr bool ACTOR = NET == NET_ACTOR;
    extern __shared__ __align__(128) unsigned char smem[];
    __shared__ __align__(8) unsigned long long mma_bar, slot_bars[2];
    __shared__ unsigned tmem_base_slot;
    __shared__ unsigned long long s_call;
    const int row = threadIdx.x, c = blockIdx.y;
    const long tile = blockIdx.x;
    const unsigned bar = (unsigned)__cvta_generic_to_shared(&mma_bar);
    const unsigned sbar0 = (unsigned)__cvta_generic_to_shared(&slot_bars[0]), sbar1 = (unsigned)__cvta_generic_to_shared(&slot_bars[1]);
    auto sbar = [&](int l) { return (l & 1) ? sbar1 : sbar0; };
    if (row == 0) {
        mbar_init(bar);
        mbar_init(sbar0);
        mbar_init(sbar1);
        fence_mbar_init();
        if constexpr (ACTOR) s_call = device_call_number(&a.calls[0], &a.calls[1]);
    }
    tmem_cta_alloc<H>(&tmem_base_slot);
    crit::CriticArgs ca{};
    ca.actor = a.net; ca.critic = a.net; ca.nqp = a.nqp;
    const int g0 = ACTOR ? 0 : 4 + 4 * c;   // the network's first layer in layer_of's sequence
    auto load_layer = [&](int l) {   // thread 0: layer l of the network -> slot l % 2
        const crit::Layer L = crit::layer_of(ca, g0 + l);
        if constexpr (ACTOR) {   // the actor's hidden biases are a separate region of its block
            mbar_expect_tx(sbar(l), (unsigned)(L.bytes0 + L.bytes1));
            if (L.src1) bulk_copy(smem + (l & 1) * crit::SLOT_BYTES + L.bytes0, L.src1, (unsigned)L.bytes1, sbar(l));
        } else {
            mbar_expect_tx(sbar(l), (unsigned)L.bytes0);
        }
        bulk_copy(smem + (l & 1) * crit::SLOT_BYTES, L.src0, (unsigned)L.bytes0, sbar(l));
    };
    if (row == 0) { load_layer(0); load_layer(1); }
    const unsigned tmem_d = tmem_base_slot;
    const unsigned tmem_row = tmem_d + ((unsigned)(row & ~31) << 16);
    const unsigned smem_base = (unsigned)__cvta_generic_to_shared(smem);
    const unsigned a_hi = smem_base + crit::OFF_A, a_lo = a_hi + A_BYTES;
    unsigned char* a_row16 = smem + crit::OFF_A + (row >> 3) * (KIN / 8 * 128) + (row & 7) * 16;
    unsigned char* a_row128 = smem + crit::OFF_A + (row >> 3) * (H / 8 * 128) + (row & 7) * 16;
    *reinterpret_cast<uint4*>(smem + crit::OFF_ONES + (row >> 3) * 256 + (row & 7) * 16) = make_uint4(0x3f803f80u, 0x3f80u, 0u, 0u);
    *reinterpret_cast<uint4*>(smem + crit::OFF_ONES + (row >> 3) * 256 + (row & 7) * 16 + 128) = make_uint4(0u, 0u, 0u, 0u);
    const long r = tile * TM + row;
    const bool ok = r < a.n;
    float x[KIN];
    load_obs_act(a.obs, a.act, a.obs_dim, ACTOR ? 0 : a.act_dim, r, ok, x);   // the actor's input is obs alone (act_dim: its head's)
    put_split_row16(a_row16, x);
    // the actor's eps: stream 11, counter (row, call lo, call hi, 11 * 65536 + pair) as the critic target's stream 10
    float2 eps[NOUT / 2];
    if constexpr (ACTOR) {
        const unsigned long long call = s_call;
#pragma unroll
        for (int pr = 0; pr < NOUT / 2; ++pr)
            eps[pr] = (ok && 2 * pr < a.act_dim)
                          ? normal_pair(a.seed, (unsigned long long)(unsigned)r | (call << 32), (unsigned)(call >> 32), (unsigned)pr, STREAM_ACTOR_GRAD)
                          : make_float2(0.0f, 0.0f);
    }
    unsigned parity = 0;
#pragma unroll 1
    for (int l = 0; l < 4; ++l) {
        publish();
        if (row == 0) {
            const crit::Layer L = crit::layer_of(ca, g0 + l);
            mbar_wait(sbar(l), (unsigned)(l >> 1));
            const unsigned slot = smem_base + (unsigned)((l & 1) * crit::SLOT_BYTES);
            issue_split_layer(tmem_d, a_hi, a_lo, slot, (unsigned)L.w_bytes, L.K, L.N, ACTOR ? L.bias : true, slot + 2 * L.w_bytes,
                              smem_base + crit::OFF_ONES, bar);
        }
        mbar_wait(bar, parity);
        parity ^= 1u;
        tc_fence_after();
        if (row == 0 && l + 2 < 4) load_layer(l + 2);
        if (l < 3) {
            if (a.saved) {   // z_l of this row, feature-major inside the tile
                float* z = a.saved + (((long)c * 3 + l) * a.n_tiles + tile) * (H * TM) + row;
                for_acc_chunks(tmem_row, [&](const unsigned (&w)[16], int c0) {
#pragma unroll
                    for (int e = 0; e < 16; ++e) z[(c0 + e) * TM] = __uint_as_float(w[e]);
                });
            }
            gelu_split_row(tmem_row, a_row128);
        } else if constexpr (ACTOR) {
            // the squashed head (b4 = b_mu[8] then b_log_std[8]); head_pair writes action column k of row r at
            // act[k * ld + 0]: act = this row of actions, ld = 1
            const float* b4 = reinterpret_cast<const float*>(a.net + f32::OFF_B) + 3 * H;
            PolicyArgs pa{};
            pa.act = a.actions + r * a.act_dim; pa.eps = a.eps ? a.eps + r * a.act_dim : nullptr; pa.ld = 1; pa.act_dim = a.act_dim;
            const float2 no_noise[NOUT / 2] = {};
            const float lp = head_row<HEAD_SQUASHED, true>(pa, tmem_row, b4, eps, no_noise, 0, ok);
            if (ok) a.logp[r] = lp + a.logp_const;
            if (a.saved) {   // head_pair's mu and log_std pre-activation (the same fp32 additions) and eps
                unsigned hv[16];
                tmem_ld16(tmem_row, hv);
                tmem_wait_ld();
                float* s = a.saved + head_saved_offset(a.n_tiles) + tile * (3 * NOUT * TM) + row;
#pragma unroll
                for (int k = 0; k < NOUT; ++k) {
                    s[k * TM] = __uint_as_float(hv[k]) + b4[k];
                    s[(NOUT + k) * TM] = __uint_as_float(hv[NOUT + k]) + b4[NOUT + k];
                    s[(2 * NOUT + k) * TM] = k & 1 ? eps[k >> 1].y : eps[k >> 1].x;
                }
            }
        } else {
            float* q = a.q + (r * a.nc + c) * a.nq;
#pragma unroll 1
            for (int h = 0; h < a.nqp; h += 16) {
                unsigned v[16];
                tmem_ld16(tmem_row + (unsigned)h, v);
                tmem_wait_ld();
#pragma unroll
                for (int e = 0; e < 16; ++e)
                    if (ok && h + e < a.nq) q[h + e] = __uint_as_float(v[e]);
            }
        }
    }
    tmem_cta_free<H>(tmem_d);
}

// torch's GELU backward (erf form): d gelu / dz = cdf(z) + z pdf(z)
__device__ __forceinline__ float gelu_erf_grad(float z) {
    const float cdf = 0.5f * (1.0f + erff(z * 0.707106781186547524f));
    const float pdf = expf(-0.5f * z * z) * 0.398942280401432678f;
    return fmaf(z, pdf, cdf);
}
// 8 fp32 values -> one 16-byte hi chunk at dst and its lo chunk A_BYTES after it
__device__ __forceinline__ void put_split8(unsigned char* dst, const float (&v)[8]) {
    unsigned hi[4], lo[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) split_pack2(v[2 * e], v[2 * e + 1], hi[e], lo[e]);
    *reinterpret_cast<uint4*>(dst) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
    *reinterpret_cast<uint4*>(dst + A_BYTES) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
}
// an operand of a split product: hi / lo start addresses, the strides between core matrices along K (the descriptor's
// leading byte offset) and along M or N (its stride byte offset) - the same two fields for K-major and MN-major operands -
// and the byte advance per K = 16 step
struct SplitOp { unsigned hi, lo, k_stride, mn_stride, step; };
// D[128 x N] (+)= A[128 x K] B[N x K]^T as issue_split_layer's three products per K = 16 step, for operands of either
// major-ness (idesc carries the transpose bits); B.lo == 0: B is exact in bf16 (the ones block), two products
__device__ __forceinline__ void issue_split_mma(unsigned d, SplitOp A, SplitOp B, unsigned idesc, int ksteps, bool accumulate) {
    const unsigned long long ah = smem_desc(A.hi, A.k_stride, A.mn_stride), al = smem_desc(A.lo, A.k_stride, A.mn_stride);
    const unsigned long long bh = smem_desc(B.hi, B.k_stride, B.mn_stride), bl = smem_desc(B.lo, B.k_stride, B.mn_stride);
    for (int j = 0; j < ksteps; ++j) {
        const unsigned long long oa = (unsigned long long)((j * A.step) >> 4), ob = (unsigned long long)((j * B.step) >> 4);
        mma_ss(d, ah + oa, bh + ob, idesc, (accumulate || j > 0) ? 1u : 0u);
        mma_ss(d, al + oa, bh + ob, idesc, 1u);
        if (B.lo) mma_ss(d, ah + oa, bl + ob, idesc, 1u);
    }
}
constexpr unsigned A_MN = 1u << 15, B_MN = 1u << 16;   // instruction descriptor: A / B read MN-major

struct BwdArgs {
    const unsigned char* net;          // as FwdArgs::net
    long n, n_tiles, tpc;              // tpc: tiles per CTA
    const float *obs, *act, *saved, *grad_q;
    float* part;                       // [nc][gridDim.x][part_floats(nqp)]; null: no weight gradients
    float* gact;                       // [nc][n][act_dim]; null: no action gradient
    int obs_dim, act_dim, nc, nq, nqp;
    // the actor (act_dim = 0: its input is obs alone; nqp = HEAD_N): d loss / d actions [n][head_dim] and d loss / d log_prob
    // [n], each nullable
    const float *grad_actions, *grad_logp;
    int head_dim;
};

// dZ of the squashed head for row r (zeros past n and head_dim): from a = tanh(x), x = mu + exp(ls) eps, ls = clamp(ls_pre,
// -20, 2) recomputed as squash() computes them (bit for bit) and SB3's log-prob,
//   g_x = g_a (1 - a^2) + g_lp 2a (1 - a^2) / (1 - a^2 + 1e-6),   g_mu = g_x,
//   g_ls_pre = (g_x exp(ls) eps - g_lp) [-20 <= ls_pre <= 2]
// (the Normal term's two paths to mu cancel; torch's clamp passes the gradient at the bounds).  dz[k] = g_mu of column k,
// dz[NOUT + k] = g_ls_pre; s = this row's saved head values (feature j at s[j * TM])
__device__ __forceinline__ void actor_head_dz(const BwdArgs& a, const float* s, long r, bool ok, float (&dz)[2 * NOUT]) {
    const float glp = (ok && a.grad_logp) ? a.grad_logp[r] : 0.0f;
#pragma unroll
    for (int k = 0; k < NOUT; ++k) {
        const bool valid = ok && k < a.head_dim;
        const float mu = s[k * TM], ls_pre = s[(NOUT + k) * TM], e = s[(2 * NOUT + k) * TM];
        const float ga = (valid && a.grad_actions) ? a.grad_actions[r * a.head_dim + k] : 0.0f;
        const float sd = expf(fminf(2.0f, fmaxf(-20.0f, ls_pre)));
        const float act = tanhf(fmaf(sd, e, mu));
        const float om = fmaf(-act, act, 1.0f);
        const float gx = fmaf(ga, om, glp * (2.0f * act) * om / (om + 1e-6f));
        dz[k] = valid ? gx : 0.0f;
        dz[NOUT + k] = (valid && ls_pre >= -20.0f && ls_pre <= 2.0f) ? fmaf(gx * sd, e, -glp) : 0.0f;
    }
}

template <int NET>
__global__ void __launch_bounds__(TM, 1) critic_backward_kernel(const __grid_constant__ BwdArgs a) {
    constexpr bool ACTOR = NET == NET_ACTOR;
    extern __shared__ __align__(128) unsigned char smem[];
    __shared__ __align__(8) unsigned long long mma_bar, slot_bar;
    __shared__ unsigned tmem_base_slot;
    const int row = threadIdx.x, c = blockIdx.y;
    const bool want_w = a.part != nullptr;
    const unsigned bar = (unsigned)__cvta_generic_to_shared(&mma_bar), sbar = (unsigned)__cvta_generic_to_shared(&slot_bar);
    if (row == 0) {
        mbar_init(bar);
        mbar_init(sbar);
        fence_mbar_init();
    }
    tmem_cta_alloc<BWD_TMEM_COLS>(&tmem_base_slot);
    const long t0 = (long)blockIdx.x * a.tpc, t1 = t0 + a.tpc < a.n_tiles ? t0 + a.tpc : a.n_tiles;
    const unsigned char* cb = a.net + (long)c * crit::critic_bytes(a.nqp);
    // weights hi, lo of layer l (0..3) of this network: its place in the network's block and bytes of one of hi / lo
    auto w_src = [&](int l) {
        if constexpr (ACTOR) return a.net + (l == 0 ? f32::OFF_W1 : l == 1 ? f32::OFF_W2 : l == 2 ? f32::OFF_W3 : f32::OFF_W4);
        else return cb + (l == 0 ? 0 : crit::L1_BYTES + (l - 1) * crit::LH_BYTES);
    };
    auto w_bytes = [&](int l) { return l == 0 ? f32::W1_BYTES : l < 3 ? f32::WH_BYTES : a.nqp * H * 2; };
    unsigned slot_parity = 0;
    auto load_w = [&](int l) {   // thread 0, once the slot's MMAs have completed
        mbar_expect_tx(sbar, (unsigned)(2 * w_bytes(l)));
        bulk_copy(smem + B_OFF_W, w_src(l), (unsigned)(2 * w_bytes(l)), sbar);
    };
    if (row == 0 && t0 < t1) load_w(3);
    const unsigned tmem = tmem_base_slot;
    const unsigned tmem_row = tmem + ((unsigned)(row & ~31) << 16);
    const unsigned sb = (unsigned)__cvta_generic_to_shared(smem);
    *reinterpret_cast<uint4*>(smem + B_OFF_ONES + (row >> 3) * 256 + (row & 7) * 16) = make_uint4(0x3f803f80u, 0x3f80u, 0u, 0u);
    *reinterpret_cast<uint4*>(smem + B_OFF_ONES + (row >> 3) * 256 + (row & 7) * 16 + 128) = make_uint4(0u, 0u, 0u, 0u);
    unsigned char* dz_row128 = smem + B_OFF_DZ + (row >> 3) * (H / 8 * 128) + (row & 7) * 16;
    unsigned char* h_row128 = smem + B_OFF_H + (row >> 3) * (H / 8 * 128) + (row & 7) * 16;
    unsigned char* h_row16 = smem + B_OFF_H + (row >> 3) * (KIN / 8 * 128) + (row & 7) * 16;
    const int nq8 = a.nqp / 8;
    unsigned char* dz_rowq = smem + B_OFF_DZ + (row >> 3) * (nq8 * 128) + (row & 7) * 16;
    // operands.  K-major tiles written row by row: K-direction stride 128, MN-direction (K / 8) 128, advance 256 per K step.
    // The same tiles read MN-major (rows = K): MN-direction stride 128, K-direction (row group) (width / 8) 128, advance twice that.
    const SplitOp dz_k = {sb + B_OFF_DZ, sb + B_OFF_DZ + A_BYTES, 128u, (unsigned)H / 8 * 128u, 256u};
    const SplitOp dzq_k = {sb + B_OFF_DZ, sb + B_OFF_DZ + A_BYTES, 128u, (unsigned)nq8 * 128u, 256u};
    const SplitOp dz_mn = {sb + B_OFF_DZ, sb + B_OFF_DZ + A_BYTES, (unsigned)H / 8 * 128u, 128u, 2u * H / 8 * 128u};
    const SplitOp dzq_mn = {sb + B_OFF_DZ, sb + B_OFF_DZ + A_BYTES, (unsigned)nq8 * 128u, 128u, 2u * nq8 * 128u};
    const SplitOp h_mn = {sb + B_OFF_H, sb + B_OFF_H + A_BYTES, (unsigned)H / 8 * 128u, 128u, 2u * H / 8 * 128u};
    const SplitOp x_mn = {sb + B_OFF_H, sb + B_OFF_H + A_BYTES, (unsigned)KIN / 8 * 128u, 128u, 2u * KIN / 8 * 128u};
    const SplitOp ones_mn = {sb + B_OFF_ONES, 0u, (unsigned)KIN / 8 * 128u, 128u, 2u * KIN / 8 * 128u};
    // the packed W [out][in] (canonical K-major, K = in) as the B operand W^T of a dgrad: N = in, K = out, read MN-major
    auto w_mn = [&](int l) {
        const unsigned kin = l == 0 ? KIN : H;
        return SplitOp{sb + B_OFF_W, sb + B_OFF_W + (unsigned)w_bytes(l), kin / 8 * 128u, 128u, 2u * kin / 8 * 128u};
    };
    float db4[crit::MAX_QUANTILES];
#pragma unroll
    for (int q = 0; q < crit::MAX_QUANTILES; ++q) db4[q] = 0.0f;
    unsigned parity = 0;
    // z_l (l = 0, 1, 2) of this row: feature j at z[j * TM]
    auto zrow = [&](int l, long tile) { return a.saved + (((long)c * 3 + l) * a.n_tiles + tile) * (H * TM) + row; };
    // H = gelu(z) of this row, split, into the H tile (K = 128 layout)
    auto put_h = [&](const float* z) {
#pragma unroll 2
        for (int j8 = 0; j8 < H / 8; ++j8) {
            float v[8];
#pragma unroll
            for (int e = 0; e < 8; ++e) v[e] = gelu_erf(z[(8 * j8 + e) * TM]);
            put_split8(h_row128 + j8 * 128, v);
        }
    };
    // dZ = dH GELU'(z) of this row (dH: the layer accumulator), split, into the dZ tile (K = 128 layout)
    auto put_dz = [&](const float* z) {
        for_acc_chunks(tmem_row + T_ACC, [&](const unsigned (&w)[16], int c0) {
#pragma unroll
            for (int q = 0; q < 2; ++q) {
                float v[8];
#pragma unroll
                for (int e = 0; e < 8; ++e) v[e] = __uint_as_float(w[8 * q + e]) * gelu_erf_grad(z[(c0 + 8 * q + e) * TM]);
                put_split8(dz_row128 + ((c0 >> 3) + q) * 128, v);
            }
        });
    };
    auto wait_mma = [&]() {
        mbar_wait(bar, parity);
        parity ^= 1u;
        tc_fence_after();
    };
    auto wait_w = [&]() {   // thread 0
        mbar_wait(sbar, slot_parity);
        slot_parity ^= 1u;
    };
    const unsigned id_dgrad = instr_desc(TM, H) | B_MN, id_dgrad1 = instr_desc(TM, KIN) | B_MN;
    const unsigned id_w = instr_desc(TM, H) | A_MN | B_MN, id_w16 = instr_desc(TM, 16) | A_MN | B_MN;
    const unsigned id_w4 = instr_desc(TM, a.nqp) | A_MN | B_MN;
#pragma unroll 1
    for (long tile = t0; tile < t1; ++tile) {
        const long r = tile * TM + row;
        const bool ok = r < a.n;
        const bool acc = tile > t0;
        // ---- output layer: dZ4 = grad_q of this row (zeros past n and nq), or the actor's dZ_head; H3 = gelu(z3)
        if constexpr (ACTOR) {
            float dz[2 * NOUT];
            actor_head_dz(a, a.saved + head_saved_offset(a.n_tiles) + tile * (3 * NOUT * TM) + row, r, ok, dz);
#pragma unroll
            for (int q8 = 0; q8 < 2; ++q8) {
                float v[8];
#pragma unroll
                for (int e = 0; e < 8; ++e) {
                    v[e] = dz[8 * q8 + e];
                    db4[8 * q8 + e] += v[e];   // the head biases: a fixed-order sum per row
                }
                put_split8(dz_rowq + q8 * 128, v);
            }
            if (want_w) put_h(zrow(2, tile));
        } else {
            const float* g = a.grad_q + (r * a.nc + c) * a.nq;
            for (int q8 = 0; q8 < nq8; ++q8) {
                float v[8];
#pragma unroll
                for (int e = 0; e < 8; ++e) v[e] = (ok && 8 * q8 + e < a.nq) ? g[8 * q8 + e] : 0.0f;
                put_split8(dz_rowq + q8 * 128, v);
#pragma unroll
                for (int e = 0; e < 8; ++e) {   // the output bias: a fixed-order sum per row, constant indices into db4
#pragma unroll
                    for (int qq = 0; qq < crit::MAX_QUANTILES / 8; ++qq)
                        if (qq == q8) db4[8 * qq + e] += v[e];
                }
            }
            if (want_w) put_h(zrow(2, tile));
        }
        publish();
        if (row == 0) {
            wait_w();
            issue_split_mma(tmem + T_ACC, dzq_k, w_mn(3), id_dgrad, a.nqp / 16, false);             // dH3 = dZ4 W4
            if (want_w) issue_split_mma(tmem + T_W4, h_mn, dzq_mn, id_w4, TM / 16, acc);              // dW4^T += H3^T dZ4
            mma_commit(bar);
        }
        wait_mma();
        // ---- hidden layers l = 2, 1, 0 (W3, W2, W1 in the slot): dZ_{l+1} = dH GELU'(z_{l+1}), then dgrad and wgrad of layer l
#pragma unroll 1
        for (int l = 2; l >= 0; --l) {
            if (row == 0) load_w(l);
            put_dz(zrow(l, tile));
            if (want_w) {
                if (l > 0) put_h(zrow(l - 1, tile));
                else {
                    float x[KIN];
                    load_obs_act(a.obs, a.act, a.obs_dim, a.act_dim, r, ok, x);
                    put_split_row16(h_row16, x);
                }
            }
            publish();
            if (row == 0) {
                wait_w();
                if (l > 0) issue_split_mma(tmem + T_ACC, dz_k, w_mn(l), id_dgrad, H / 16, false);          // dH_{l-1} = dZ_l W_l
                else if (a.gact) issue_split_mma(tmem + T_ACC, dz_k, w_mn(0), id_dgrad1, H / 16, false);   // d[obs, act] = dZ1 W1
                if (want_w) {
                    const unsigned tw = l == 2 ? T_W3 : l == 1 ? T_W2 : T_W1, tb = l == 2 ? T_B3 : l == 1 ? T_B2 : T_B1;
                    if (l > 0) issue_split_mma(tmem + tw, dz_mn, h_mn, id_w, TM / 16, acc);       // dW += dZ^T H
                    else issue_split_mma(tmem + tw, dz_mn, x_mn, id_w16, TM / 16, acc);           // dW1 += dZ1^T [obs, act]
                    issue_split_mma(tmem + tb, dz_mn, ones_mn, id_w16, TM / 16, acc);                              // db += dZ^T 1
                }
                mma_commit(bar);
            }
            wait_mma();
        }
        if (row == 0 && tile + 1 < t1) load_w(3);
        // ---- the action columns of d[obs, act] (this critic's part)
        if (a.gact) {
            unsigned v[16];
            tmem_ld16(tmem_row + T_ACC, v);
            tmem_wait_ld();
#pragma unroll
            for (int j = 0; j < KIN; ++j) {   // column j = action k (constant indices into v)
                const int k = j - a.obs_dim;
                if (ok && k >= 0 && k < a.act_dim) a.gact[((long)c * a.n + r) * a.act_dim + k] = __uint_as_float(v[j]);
            }
        }
    }
    // ---- this CTA's partial of every parameter gradient: TMEM T_W1 .. T_W4 + nqp lane-major, then the output bias
    if (want_w && t0 < t1) {
        float* part = a.part + ((long)c * gridDim.x + blockIdx.x) * part_floats(a.nqp);
        const int ncol = T_W4 - T_W1 + a.nqp;
#pragma unroll 1
        for (int c0 = 0; c0 < ncol; c0 += 16) {
            unsigned v[16];
            tmem_ld16(tmem_row + (unsigned)(T_W1 + c0), v);
            tmem_wait_ld();
#pragma unroll
            for (int e = 0; e < 16; ++e) part[(long)(c0 + e) * TM + row] = __uint_as_float(v[e]);
        }
        float* s = reinterpret_cast<float*>(smem + B_OFF_H);   // every MMA has completed: the H tile is free
        constexpr int LD = crit::MAX_QUANTILES + 1;
#pragma unroll
        for (int q = 0; q < crit::MAX_QUANTILES; ++q) s[row * LD + q] = db4[q];
        __syncthreads();
        if (row < a.nqp) {
            float sum = 0.0f;
            for (int i = 0; i < TM; ++i) sum += s[i * LD + row];
            part[(long)ncol * TM + row] = sum;
        }
    }
    tmem_cta_free<BWD_TMEM_COLS>(tmem);
}

struct ReduceArgs {
    const float *part, *gact;
    float* grads[MAX_CRITICS * 8];     // nn.Linear layout; grads[0] null: none
    float* grad_act;                   // [n][act_dim], nullable
    long n;
    int nc, nq, nqp, k, act_dim, ctas;
};
constexpr int REDUCE_THREADS = 256;

// one thread per word of a partial block (then per element of grad_act): the sum over the CTAs of a critic in CTA order,
// stored at the parameter's place; grad_act = the sum over the critics in critic order.  The actor (nc = 1, nq = act_dim,
// grads in squashed_param_shapes order): dW_head^T columns 0..act_dim-1 are mu.weight's rows, 8..8+act_dim-1 log_std.weight's
template <int NET>
__global__ void __launch_bounds__(REDUCE_THREADS) critic_grad_reduce_kernel(const __grid_constant__ ReduceArgs a) {
    const long i = (long)blockIdx.x * REDUCE_THREADS + threadIdx.x;
    const long pf = part_floats(a.nqp), nw = a.grads[0] ? (long)a.nc * pf : 0;
    if (i < nw) {
        const int c = (int)(i / pf);
        const long w = i % pf;
        const int col = (int)(w / TM) + T_W1, lane = (int)(w % TM);
        const long bias4 = (long)(T_W4 - T_W1 + a.nqp) * TM;
        float* dst = nullptr;
        if (NET == NET_ACTOR && (w >= bias4 || col >= T_W4)) {   // the squashed head: mu in columns 0..7, log_std in 8..15
            const int j = w >= bias4 ? (int)(w - bias4) : col - T_W4, k = j % NOUT;
            if (j < 2 * NOUT && k < a.nq)
                dst = w >= bias4 ? a.grads[j < NOUT ? 7 : 9] + k : a.grads[j < NOUT ? 6 : 8] + k * H + lane;
        }
        else if (w >= bias4) { if (w - bias4 < a.nq) dst = a.grads[8 * c + 7] + (w - bias4); }   // the output bias
        else if (col < T_B1) { if (col - T_W1 < a.k) dst = a.grads[8 * c + 0] + lane * a.k + (col - T_W1); }
        else if (col < T_W2) { if (col == T_B1) dst = a.grads[8 * c + 1] + lane; }
        else if (col < T_B2) dst = a.grads[8 * c + 2] + lane * H + (col - T_W2);
        else if (col < T_W3) { if (col == T_B2) dst = a.grads[8 * c + 3] + lane; }
        else if (col < T_B3) dst = a.grads[8 * c + 4] + lane * H + (col - T_W3);
        else if (col < T_W4) { if (col == T_B3) dst = a.grads[8 * c + 5] + lane; }
        else if (col - T_W4 < a.nq) dst = a.grads[8 * c + 6] + (col - T_W4) * H + lane;   // dW4^T: lane = input feature
        if (!dst) return;
        const float* p = a.part + (long)c * a.ctas * pf + w;
        float sum = 0.0f;
        for (int j = 0; j < a.ctas; ++j) sum += p[(long)j * pf];
        *dst = sum;
        return;
    }
    const long e = i - nw;
    if (!a.grad_act || e >= a.n * a.act_dim) return;
    float sum = 0.0f;
    for (int c = 0; c < a.nc; ++c) sum += a.gact[(long)c * a.n * a.act_dim + e];
    a.grad_act[e] = sum;
}

}  // namespace cgrad

// =====================================================================================================================
// Weight packing: ONE kernel writes a handle's whole parameter block(s) from fp32 arrays in device memory (torch.nn.Linear
// layout, W [out][in]), on the caller's stream.  The learner's CUDA tensors are read where they are (no host copy, no
// synchronisation, capturable in a CUDA graph); the host entries stage their arrays into a per-handle device buffer and run
// the same kernel.  One thread per 4-byte output word: every word of every block is rewritten on each call, padding
// (obs_dim < 16, act_dim < 8, unused head rows) as zeros.  The sources are read one float at a time, so a tensor with a
// storage offset (4-byte alignment only) is fine.
//
// The bytes are the ones the library has always packed (it packed on the host before), for every input, Inf and NaN
// included: bf16 rounding by bf16_bits (round to nearest even on the bits; a NaN keeps its upper half with the quiet bit set,
// which __float2bfloat16_rn does not do), and the fp32 operations of the packing (the 0.5 scale of the tcgen05 weights, the
// subtractions of the hi / lo and bias-term splits) with the NaN results of x86-64 SSE arithmetic (sub_x86, mul_x86).
// =====================================================================================================================
struct PackSrc {   // v0 / v1 [act_dim] fill the b4 / std slots (fixed: b4, exp(log_std); squashed: b_mu, b_log_std)
    const float *W1, *b1, *W2, *b2, *W3, *b3, *W4, *v0, *Wls, *v1;   // Wls: the squashed head's log_std layer, NULL for the fixed head
};
struct PackArgs {
    PackSrc s;
    unsigned* frag;      // mma.sync B-fragment block (bf16 handles; NULL for fp32 handles)
    unsigned* canon;     // tcgen05 block: canonical K-major (bf16 handles) or the split hi / lo block (fp32 handles)
    int frag_words, canon_words, obs_dim, act_dim, fp32;
    // critic handles (frag_words = canon_words = 0): n_critics blocks of crit::critic_bytes(nqp) from W1 b1 W2 b2 W3 b3 W4 b4
    // of each critic; W1 [128][critic_k], W4 [nq][128]
    unsigned* critic;
    int critic_words, critic_k, critic_nq, critic_nqp;
    const float* cw[crit::MAX_CRITICS * 8];
};
constexpr int PACK_THREADS = 256;

__device__ __forceinline__ unsigned bf16_bits(float f) {   // round to nearest even, like __float2bfloat16_rn; NaN: quiet, upper half kept
    unsigned u = __float_as_uint(f);
    if ((u & 0x7fffffffu) > 0x7f800000u) return (u >> 16) | 0x40u;
    u += 0x7fffu + ((u >> 16) & 1u);
    return u >> 16;
}
__device__ __forceinline__ float bf16_value(float f) { return __uint_as_float(bf16_bits(f) << 16); }
__device__ __forceinline__ bool is_nan(float f) { return (__float_as_uint(f) & 0x7fffffffu) > 0x7f800000u; }
__device__ __forceinline__ float quiet(float f) { return __uint_as_float(__float_as_uint(f) | 0x400000u); }
// a - b as SSE subss computes it: a NaN operand comes back quieted (the first one if both are), Inf - Inf is the default NaN
// 0xffc00000 (the GPU's subtraction returns 0x7fffffff for all three)
__device__ __forceinline__ float sub_x86(float a, float b) {
    if (is_nan(a)) return quiet(a);
    if (is_nan(b)) return quiet(b);
    const float r = __fsub_rn(a, b);
    return is_nan(r) ? __uint_as_float(0xffc00000u) : r;
}
__device__ __forceinline__ float mul_x86(float s, float w) { return is_nan(w) ? quiet(w) : __fmul_rn(s, w); }   // s finite, non-zero

enum PackOp { OP_BF16, OP_HALF, OP_LO };   // bf16 of w, of 0.5 w (the tcgen05 layers that read doubled activations), of w - bf16(w)
// bf16 bits of element (n, k) of W [N][K] under `op`; 0 outside N x K
__device__ __forceinline__ unsigned w_elem(const float* W, int N, int K, int n, int k, PackOp op) {
    if (n >= N || k >= K) return 0u;
    const float w = W[(size_t)n * K + k];
    if (op == OP_HALF) return bf16_bits(mul_x86(0.5f, w));
    if (op == OP_LO) return bf16_bits(sub_x86(w, bf16_value(w)));
    return bf16_bits(w);
}
// the head block [16 x 128]: the first head layer in rows 0..act_dim-1, the squashed head's log_std layer in rows 8..8+act_dim-1
__device__ __forceinline__ unsigned head_elem(const PackArgs& p, int n, int k, PackOp op) {
    return n < NOUT ? w_elem(p.s.W4, p.act_dim, H, n, k, op) : (p.s.Wls ? w_elem(p.s.Wls, p.act_dim, H, n - NOUT, k, op) : 0u);
}
// float b1[128] b2[128] b3[128] b4[8] std[8], as bits
__device__ __forceinline__ unsigned bias_slot(const PackArgs& p, int f) {
    if (f < 3 * H) return __float_as_uint((f < H ? p.s.b1 : f < 2 * H ? p.s.b2 : p.s.b3)[f % H]);
    const int k = (f - 3 * H) % NOUT;
    return k < p.act_dim ? __float_as_uint((f < 3 * H + NOUT ? p.s.v0 : p.s.v1)[k]) : 0u;
}
// term t of the bias split b = t0 + t1 + t2 (every term a bf16) of the bias-MMA blocks
__device__ __forceinline__ unsigned bias_term(float b, int t) {
    for (int j = 0; j < t; ++j) b = sub_x86(b, bf16_value(b));
    return bf16_bits(b);
}

// word i of the mma.sync block: for k-step kk, n-tile nt, lane (g = lane / 4, t = lane % 4) the two uint32 of the B fragment,
// (W[8 nt + g][16 kk + 2t], +1) and (W[8 nt + g][16 kk + 8 + 2t], +1)
__device__ unsigned frag_word(const PackArgs& p, int i) {
    const int off = 4 * i;
    if (off >= OFF_B && off < PACKED_BYTES) return bias_slot(p, (off - OFF_B) / 4);
    const float* W = p.s.W2;
    int N = H, K = H, n_tiles = 16, base = OFF_W2;
    if (off < OFF_W2) { W = p.s.W1; K = p.obs_dim; base = OFF_W1; }
    else if (off >= OFF_W3 && off < OFF_W4) { W = p.s.W3; base = OFF_W3; }
    else if (off >= OFF_W4) { W = off < OFF_B ? p.s.W4 : p.s.Wls; N = p.act_dim; n_tiles = 1; base = off < OFF_B ? OFF_W4 : OFF_WLS; }
    const int j = (off - base) / 4, lane = (j >> 1) & 31, q = j >> 6;
    const int n = 8 * (q % n_tiles) + (lane >> 2), k = 16 * (q / n_tiles) + 2 * (lane & 3) + 8 * (j & 1);
    return w_elem(W, N, K, n, k, OP_BF16) | (w_elem(W, N, K, n, k + 1, OP_BF16) << 16);
}

// (n, k) of the bf16 pair at byte offset `rel` of an [Np x Kp] canonical K-major matrix: element (n, k) sits at bf16 index
// ((n / 8) (Kp / 8) + k / 8) 64 + (n % 8) 8 + k % 8
__device__ __forceinline__ void canon_nk(int rel, int Kp, int& n, int& k) {
    const int e = rel / 2, c = e >> 6, r = e & 63;
    n = (c / (Kp / 8)) * 8 + (r >> 3);
    k = (c % (Kp / 8)) * 8 + (r & 7);
}
// the bias-MMA blocks (three [128 x 16]: columns 0..2 = the terms of b1, b2, b3) and the ones block ([128 x 16], columns 0..2 = 1)
__device__ unsigned bias_mma_word(const PackArgs& p, int rel) {
    constexpr int BLK = H * KIN * 2;
    const int l = rel / BLK;
    int n, k;
    canon_nk(rel % BLK, KIN, n, k);
    auto elem = [&](int c) -> unsigned {
        if (c >= 3) return 0u;
        return l == 3 ? 0x3f80u : bias_term((l == 0 ? p.s.b1 : l == 1 ? p.s.b2 : p.s.b3)[n], c);
    };
    return elem(k) | (elem(k + 1) << 16);
}

// word i of the tcgen05 block of a bf16 handle: W1 as is, W2 / W3 / head scaled by 0.5 (the activations are stored doubled),
// then the bias-MMA blocks
__device__ unsigned tc5_word(const PackArgs& p, int i) {
    const int off = 4 * i;
    if (off >= tc5::OFF_BIAS) return bias_mma_word(p, off - tc5::OFF_BIAS);
    if (off >= tc5::OFF_B) return bias_slot(p, (off - tc5::OFF_B) / 4);
    int n, k;
    if (off >= tc5::OFF_W4) {
        canon_nk(off - tc5::OFF_W4, H, n, k);
        return head_elem(p, n, k, OP_HALF) | (head_elem(p, n, k + 1, OP_HALF) << 16);
    }
    if (off < tc5::OFF_W2) {
        canon_nk(off - tc5::OFF_W1, KIN, n, k);
        return w_elem(p.s.W1, H, p.obs_dim, n, k, OP_BF16) | (w_elem(p.s.W1, H, p.obs_dim, n, k + 1, OP_BF16) << 16);
    }
    const bool l2 = off < tc5::OFF_W3;
    canon_nk(off - (l2 ? tc5::OFF_W2 : tc5::OFF_W3), H, n, k);
    const float* W = l2 ? p.s.W2 : p.s.W3;
    return w_elem(W, H, H, n, k, OP_HALF) | (w_elem(W, H, H, n, k + 1, OP_HALF) << 16);
}

// word i of the block of an fp32 handle: every weight matrix as hi = bf16(w) then lo = bf16(w - hi), no scale
__device__ unsigned f32_word(const PackArgs& p, int i) {
    const int off = 4 * i;
    if (off >= f32::OFF_BIAS) return bias_mma_word(p, off - f32::OFF_BIAS);
    if (off >= f32::OFF_B) return bias_slot(p, (off - f32::OFF_B) / 4);
    int n, k;
    if (off >= f32::OFF_W4) {
        const int rel = off - f32::OFF_W4;
        const PackOp op = rel < f32::W4_BYTES ? OP_BF16 : OP_LO;
        canon_nk(rel % f32::W4_BYTES, H, n, k);
        return head_elem(p, n, k, op) | (head_elem(p, n, k + 1, op) << 16);
    }
    const float* W;
    int K, Kp, rel, bytes;
    if (off < f32::OFF_W2) { W = p.s.W1; K = p.obs_dim; Kp = KIN; rel = off - f32::OFF_W1; bytes = f32::W1_BYTES; }
    else { const bool l2 = off < f32::OFF_W3; W = l2 ? p.s.W2 : p.s.W3; K = Kp = H; rel = off - (l2 ? f32::OFF_W2 : f32::OFF_W3); bytes = f32::WH_BYTES; }
    const PackOp op = rel < bytes ? OP_BF16 : OP_LO;
    canon_nk(rel % bytes, Kp, n, k);
    return w_elem(W, H, K, n, k, op) | (w_elem(W, H, K, n, k + 1, op) << 16);
}

// word i of a critic handle's block (crit layout): per critic and layer, hi = bf16(w), lo = bf16(w - hi), no scale, then the
// layer's bias as three bf16 terms in columns 0..2 of an [N x 16] block (bias_mma_word's split); zeros past K, N and nq
__device__ unsigned critic_word(const PackArgs& p, int i) {
    const int cb = crit::critic_bytes(p.critic_nqp), off = 4 * i, c = off / cb;
    int rel = off % cb, l, K = H, Kp = H, N = H, Np = H;
    if (rel < crit::L1_BYTES) { l = 0; K = p.critic_k; Kp = KIN; }
    else if (rel < crit::L1_BYTES + 2 * crit::LH_BYTES) { rel -= crit::L1_BYTES; l = 1 + rel / crit::LH_BYTES; rel %= crit::LH_BYTES; }
    else { rel -= crit::L1_BYTES + 2 * crit::LH_BYTES; l = 3; N = p.critic_nq; Np = p.critic_nqp; }
    const float* W = p.cw[8 * c + 2 * l];
    const float* b = p.cw[8 * c + 2 * l + 1];
    const int wb = Np * Kp * 2;
    int n, k;
    if (rel >= 2 * wb) {
        canon_nk(rel - 2 * wb, KIN, n, k);
        auto elem = [&](int t) -> unsigned { return (t < 3 && n < N) ? bias_term(b[n], t) : 0u; };
        return elem(k) | (elem(k + 1) << 16);
    }
    const PackOp op = rel < wb ? OP_BF16 : OP_LO;
    canon_nk(rel % wb, Kp, n, k);
    return w_elem(W, N, K, n, k, op) | (w_elem(W, N, K, n, k + 1, op) << 16);
}

__global__ void __launch_bounds__(PACK_THREADS) policy_pack_kernel(const __grid_constant__ PackArgs p) {
    const int i = blockIdx.x * PACK_THREADS + threadIdx.x;
    if (i < p.frag_words) p.frag[i] = frag_word(p, i);
    else if (i - p.frag_words < p.canon_words) p.canon[i - p.frag_words] = p.fp32 ? f32_word(p, i - p.frag_words) : tc5_word(p, i - p.frag_words);
    else if (i - p.frag_words - p.canon_words < p.critic_words) p.critic[i - p.frag_words - p.canon_words] = critic_word(p, i - p.frag_words - p.canon_words);
}

}  // namespace

struct MvrlPolicy {
    int device, obs_dim, act_dim, sm_count;
    int head;                // MVRL_POLICY_HEAD_*: the kernel instantiation this handle launches
    int precision;           // MVRL_POLICY_PRECISION_*: bf16 = the fast kernels, fp32 = policy_act_fp32_kernel
    unsigned char* packed;   // device: B fragments of the mma.sync kernel (bf16 handles only)
    unsigned char* packed5;  // device: canonical K-major matrices of the tcgen05 kernel (fp32 handles: the hi / lo block)
    bool mma_sync;           // MVRL_POLICY_MMA_SYNC=1: the warp-level mma.sync kernel instead of tcgen05
    bool has_weights;
    float logp_const;        // fixed head: -sum(log_std); squashed head: -act_dim log(2 pi) / 2
    bool noise;              // squashed head: action noise on
    float noise_std[NOUT];
    float* staging;          // device: the host entries' arrays, copied here for policy_pack_kernel (staging_floats)
};

// floats of the staging buffer: W1 b1 W2 b2 W3 b3 W4 v0 Wls v1, back to back (PackSrc's order)
static size_t staging_floats(int obs_dim, int act_dim) { return (size_t)H * obs_dim + 3 * H + 2 * (size_t)H * H + 2 * ((size_t)act_dim * H + act_dim); }

extern "C" MVRL_API int mvrl_policy_create_ex(MvrlPolicy** out, int device, int obs_dim, int act_dim, int head, int precision) {
    if (!out) return mvrl_fail(MVRL_EINVAL, "mvrl_policy_create: null output");
    if (obs_dim < 1 || obs_dim > KIN || act_dim < 1 || act_dim > NOUT)
        return mvrl_fail(MVRL_EINVAL, "mvrl_policy_create: obs_dim must be 1..%d and act_dim 1..%d (got %d, %d)", KIN, NOUT, obs_dim, act_dim);
    if (head != HEAD_FIXED && head != HEAD_SQUASHED)
        return mvrl_fail(MVRL_EINVAL, "mvrl_policy_create_head: unknown head %d (MVRL_POLICY_HEAD_FIXED_STD or MVRL_POLICY_HEAD_SQUASHED)", head);
    if (precision != MVRL_POLICY_PRECISION_BF16 && precision != MVRL_POLICY_PRECISION_FP32)
        return mvrl_fail(MVRL_EINVAL, "mvrl_policy_create_ex: unknown precision %d (MVRL_POLICY_PRECISION_BF16 or MVRL_POLICY_PRECISION_FP32)", precision);
    const bool fp32 = precision == MVRL_POLICY_PRECISION_FP32;
    bool mma_sync;
    { const char* e = getenv("MVRL_POLICY_MMA_SYNC"); mma_sync = (e && e[0] == '1'); }
    if (fp32 && mma_sync)
        return mvrl_fail(MVRL_EINVAL, "mvrl_policy_create_ex: MVRL_POLICY_MMA_SYNC=1 selects the bf16 mma.sync kernel; the fp32 precision has the tcgen05 kernel only");
    { const int rc = mvrl_require_device(device); if (rc != MVRL_OK) return rc; }
    MVRL_ON_DEVICE(device);
    MvrlPolicy* h = new (std::nothrow) MvrlPolicy();
    if (!h) return mvrl_fail(MVRL_EINVAL, "out of host memory");
    h->device = device; h->obs_dim = obs_dim; h->act_dim = act_dim; h->has_weights = false; h->logp_const = 0.f; h->packed = nullptr; h->packed5 = nullptr; h->staging = nullptr;
    h->head = head; h->precision = precision; h->noise = false;
    for (int k = 0; k < NOUT; ++k) h->noise_std[k] = 0.0f;
    h->mma_sync = mma_sync;
    h->sm_count = 148;
    { int v = 0; if (cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, device) == cudaSuccess && v > 0) h->sm_count = v; else cudaGetLastError(); }
    cudaError_t e = cudaSuccess;
    if (fp32) {
        e = cudaMalloc(&h->packed5, f32::PARAM_BYTES);
        if (e == cudaSuccess)
            e = head == HEAD_FIXED ? cudaFuncSetAttribute(f32::policy_act_fp32_kernel<HEAD_FIXED>, cudaFuncAttributeMaxDynamicSharedMemorySize, f32::SMEM_BYTES)
                                   : cudaFuncSetAttribute(f32::policy_act_fp32_kernel<HEAD_SQUASHED>, cudaFuncAttributeMaxDynamicSharedMemorySize, f32::SMEM_BYTES);
        if (e == cudaSuccess && head == HEAD_SQUASHED)   // mvrl_actor_forward / mvrl_actor_backward
            e = cudaFuncSetAttribute(cgrad::critic_forward_kernel<cgrad::NET_ACTOR>, cudaFuncAttributeMaxDynamicSharedMemorySize, cgrad::FWD_SMEM_BYTES);
        if (e == cudaSuccess && head == HEAD_SQUASHED)
            e = cudaFuncSetAttribute(cgrad::critic_backward_kernel<cgrad::NET_ACTOR>, cudaFuncAttributeMaxDynamicSharedMemorySize, cgrad::BWD_SMEM_BYTES);
    } else {
        e = cudaMalloc(&h->packed, packed_bytes(head));
        if (e == cudaSuccess) e = cudaMalloc(&h->packed5, tc5::PARAM_BYTES);
        if (head == HEAD_FIXED) {
            if (e == cudaSuccess) e = cudaFuncSetAttribute(policy_act_kernel<HEAD_FIXED>, cudaFuncAttributeMaxDynamicSharedMemorySize, PACKED_BYTES);
            if (e == cudaSuccess) e = cudaFuncSetAttribute(tc5::policy_act_tc5_kernel<HEAD_FIXED>, cudaFuncAttributeMaxDynamicSharedMemorySize, tc5::SMEM_BYTES);
        } else {
            if (e == cudaSuccess) e = cudaFuncSetAttribute(policy_act_kernel<HEAD_SQUASHED>, cudaFuncAttributeMaxDynamicSharedMemorySize, PACKED_BYTES_SQUASHED);
            if (e == cudaSuccess) e = cudaFuncSetAttribute(tc5::policy_act_tc5_kernel<HEAD_SQUASHED>, cudaFuncAttributeMaxDynamicSharedMemorySize, tc5::SMEM_BYTES);
        }
    }
    if (e == cudaSuccess) e = cudaMalloc(&h->staging, staging_floats(obs_dim, act_dim) * sizeof(float));
    if (e != cudaSuccess) {
        if (h->packed) cudaFree(h->packed);
        if (h->packed5) cudaFree(h->packed5);
        if (h->staging) cudaFree(h->staging);
        delete h;
        return mvrl_fail(MVRL_ECUDA, "mvrl_policy_create: %s", cudaGetErrorString(e));
    }
    *out = h;
    return MVRL_OK;
}

extern "C" MVRL_API int mvrl_policy_create_head(MvrlPolicy** out, int device, int obs_dim, int act_dim, int head) {
    return mvrl_policy_create_ex(out, device, obs_dim, act_dim, head, MVRL_POLICY_PRECISION_BF16);
}

extern "C" MVRL_API int mvrl_policy_create(MvrlPolicy** out, int device, int obs_dim, int act_dim) {
    return mvrl_policy_create_head(out, device, obs_dim, act_dim, HEAD_FIXED);
}

extern "C" MVRL_API int mvrl_policy_destroy(MvrlPolicy* h) {
    if (!h) return MVRL_OK;
    { MvrlDeviceGuard guard(h->device); cudaFree(h->packed); cudaFree(h->packed5); cudaFree(h->staging); }
    delete h;
    return MVRL_OK;
}

// Every parameter block of the handle from the device arrays of `src`: one policy_pack_kernel launch on `stream`.
static int pack_weights(MvrlPolicy* h, const PackSrc& src, cudaStream_t stream) {
    PackArgs p = {};
    p.s = src;
    p.obs_dim = h->obs_dim; p.act_dim = h->act_dim;
    p.fp32 = h->precision == MVRL_POLICY_PRECISION_FP32 ? 1 : 0;
    p.frag = p.fp32 ? nullptr : reinterpret_cast<unsigned*>(h->packed);
    p.frag_words = p.fp32 ? 0 : packed_bytes(h->head) / 4;
    p.canon = reinterpret_cast<unsigned*>(h->packed5);
    p.canon_words = (p.fp32 ? f32::PARAM_BYTES : tc5::PARAM_BYTES) / 4;
    const int words = p.frag_words + p.canon_words;
    policy_pack_kernel<<<(words + PACK_THREADS - 1) / PACK_THREADS, PACK_THREADS, 0, stream>>>(p);
    return mvrl_check_launch("policy_pack");
}

// The host entries: HOST arrays in torch.nn.Linear layout -> the staging buffer -> pack_weights on the legacy default stream,
// then synchronise.  W4 [act_dim][H] is the first head layer (fixed: the mean, squashed: mu), Wls the squashed head's log_std
// layer (NULL for the fixed head); v0 / v1 [act_dim] go to the b4 / std slots.
static int set_weights_from_host(MvrlPolicy* h, const float* W1, const float* b1, const float* W2, const float* b2, const float* W3,
                                 const float* b3, const float* W4, const float* v0, const float* Wls, const float* v1) {
    const size_t w4 = (size_t)h->act_dim * H;
    const float* host[10] = {W1, b1, W2, b2, W3, b3, W4, v0, Wls, v1};
    const size_t count[10] = {(size_t)H * h->obs_dim, H, (size_t)H * H, H, (size_t)H * H, H, w4, (size_t)h->act_dim, w4, (size_t)h->act_dim};
    const float* dev[10];
    MVRL_ON_DEVICE(h->device);
    float* at = h->staging;
    for (int i = 0; i < 10; ++i) {
        dev[i] = host[i] ? at : nullptr;
        if (host[i]) MVRL_CUDA(cudaMemcpy(at, host[i], count[i] * sizeof(float), cudaMemcpyHostToDevice));
        at += count[i];
    }
    const PackSrc src = {dev[0], dev[1], dev[2], dev[3], dev[4], dev[5], dev[6], dev[7], dev[8], dev[9]};
    const int rc = pack_weights(h, src, cudaStreamLegacy);
    if (rc != MVRL_OK) return rc;
    MVRL_CUDA(cudaStreamSynchronize(cudaStreamLegacy));
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
    const int rc = set_weights_from_host(h, W1, b1, W2, b2, W3, b3, W4, b4, nullptr, sd);
    if (rc == MVRL_OK) h->logp_const = (float)(-lsum);
    return rc;
}

// the checks of both squashed-head entries that do not look at the weights
static int check_squashed(const MvrlPolicy* h, const char* who, const float* noise_std) {
    if (h->head != HEAD_SQUASHED) return mvrl_fail(MVRL_EINVAL, "%s: the handle has the fixed-std head (mvrl_policy_set_weights)", who);
    if (noise_std)
        for (int k = 0; k < h->act_dim; ++k)
            if (!(noise_std[k] >= 0.0f && noise_std[k] < INFINITY))
                return mvrl_fail(MVRL_EINVAL, "%s: noise_std[%d] = %g is not a finite value >= 0", who, k, (double)noise_std[k]);
    return MVRL_OK;
}
static void set_squashed_noise(MvrlPolicy* h, const float* noise_std) {
    h->logp_const = (float)(-0.5 * h->act_dim * log(2.0 * M_PI));
    h->noise = noise_std != nullptr;
    for (int k = 0; k < NOUT; ++k) h->noise_std[k] = (noise_std && k < h->act_dim) ? noise_std[k] : 0.0f;
}

extern "C" MVRL_API int mvrl_policy_set_weights_squashed(MvrlPolicy* h, const float* W1, const float* b1, const float* W2, const float* b2,
                                                         const float* W3, const float* b3, const float* W_mu, const float* b_mu,
                                                         const float* W_log_std, const float* b_log_std, const float* noise_std) {
    if (!h || !W1 || !b1 || !W2 || !b2 || !W3 || !b3 || !W_mu || !b_mu || !W_log_std || !b_log_std)
        return mvrl_fail(MVRL_EINVAL, "mvrl_policy_set_weights_squashed: null argument");
    int rc = check_squashed(h, "mvrl_policy_set_weights_squashed", noise_std);
    if (rc == MVRL_OK) rc = set_weights_from_host(h, W1, b1, W2, b2, W3, b3, W_mu, b_mu, W_log_std, b_log_std);
    if (rc != MVRL_OK) return rc;
    set_squashed_noise(h, noise_std);
    return MVRL_OK;
}

extern "C" MVRL_API int mvrl_policy_set_weights_squashed_device(MvrlPolicy* h, const float* W1, const float* b1, const float* W2,
                                                                const float* b2, const float* W3, const float* b3, const float* W_mu,
                                                                const float* b_mu, const float* W_log_std, const float* b_log_std,
                                                                const float* noise_std, mvrl_stream_t stream) {
    static const char* const who = "mvrl_policy_set_weights_squashed_device";
    static const char* const names[10] = {"W1", "b1", "W2", "b2", "W3", "b3", "W_mu", "b_mu", "W_log_std", "b_log_std"};
    const PackSrc src = {W1, b1, W2, b2, W3, b3, W_mu, b_mu, W_log_std, b_log_std};
    const float* const arg[10] = {W1, b1, W2, b2, W3, b3, W_mu, b_mu, W_log_std, b_log_std};
    if (!h) return mvrl_fail(MVRL_EINVAL, "%s: null handle", who);
    for (int i = 0; i < 10; ++i)
        if (!arg[i]) return mvrl_fail(MVRL_EINVAL, "%s: null argument %s", who, names[i]);
    { const int rc = check_squashed(h, who, noise_std); if (rc != MVRL_OK) return rc; }
    { const int rc = mvrl_check_device_ptrs(h->device, arg, names, 10, who); if (rc != MVRL_OK) return rc; }
    MVRL_ON_DEVICE(h->device);
    const int rc = pack_weights(h, src, (cudaStream_t)stream);
    if (rc != MVRL_OK) return rc;
    h->has_weights = true;
    set_squashed_noise(h, noise_std);
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
    // the tcgen05 kernels: one CTA per SM (small batches: one tile per SM before a second tile group gets one)
    const unsigned grid_tc = (unsigned)(tiles < (int64_t)h->sm_count ? tiles : (int64_t)h->sm_count);
    const bool squashed = h->head == HEAD_SQUASHED;
    if (h->precision == MVRL_POLICY_PRECISION_FP32) {
        a.packed = h->packed5;
        if (squashed) f32::policy_act_fp32_kernel<HEAD_SQUASHED><<<grid_tc, TM, f32::SMEM_BYTES, (cudaStream_t)stream>>>(a);
        else f32::policy_act_fp32_kernel<HEAD_FIXED><<<grid_tc, TM, f32::SMEM_BYTES, (cudaStream_t)stream>>>(a);
    } else if (h->mma_sync) {
        if (squashed) policy_act_kernel<HEAD_SQUASHED><<<grid, THREADS, PACKED_BYTES_SQUASHED, (cudaStream_t)stream>>>(a);
        else policy_act_kernel<HEAD_FIXED><<<grid, THREADS, PACKED_BYTES, (cudaStream_t)stream>>>(a);
    } else {
        a.packed = h->packed5;
        if (squashed) tc5::policy_act_tc5_kernel<HEAD_SQUASHED><<<grid_tc, TM * tc5::GROUPS, tc5::SMEM_BYTES, (cudaStream_t)stream>>>(a);
        else tc5::policy_act_tc5_kernel<HEAD_FIXED><<<grid_tc, TM * tc5::GROUPS, tc5::SMEM_BYTES, (cudaStream_t)stream>>>(a);
    }
    return mvrl_check_launch("policy_act");
}

extern "C" MVRL_API int mvrl_policy_act(MvrlPolicy* h, int64_t n, int64_t ld, const float* obs, float* act, float* logp, float* mean,
                                        float* eps, uint64_t seed, uint64_t env_id0, uint32_t step, int deterministic, mvrl_stream_t stream) {
    return mvrl_policy_act_ex(h, n, ld, obs, act, logp, mean, nullptr, eps, seed, env_id0, step, deterministic, stream);
}

// ---------------------------------------------------------------------------------------------------- critic target (K10)
struct MvrlCritic {
    int device, obs_dim, act_dim, kind, nc, nq, nqp;
    unsigned char* packed;   // device: n_critics blocks of crit::critic_bytes(nqp)
    bool has_weights;
};

extern "C" MVRL_API int mvrl_critic_create(MvrlCritic** out, int device, int obs_dim, int act_dim, int kind, int n_critics, int n_quantiles) {
    static const char* const who = "mvrl_critic_create";
    if (!out) return mvrl_fail(MVRL_EINVAL, "%s: null output", who);
    if (obs_dim < 1 || act_dim < 1 || act_dim > NOUT || obs_dim + act_dim > KIN)
        return mvrl_fail(MVRL_EINVAL, "%s: need obs_dim >= 1, 1 <= act_dim <= %d and obs_dim + act_dim <= %d (got %d, %d)", who, NOUT, KIN, obs_dim, act_dim);
    if (kind != MVRL_CRITIC_SAC && kind != MVRL_CRITIC_TQC)
        return mvrl_fail(MVRL_EINVAL, "%s: unknown kind %d (MVRL_CRITIC_SAC or MVRL_CRITIC_TQC)", who, kind);
    if (n_critics < 1 || n_critics > crit::MAX_CRITICS)
        return mvrl_fail(MVRL_EINVAL, "%s: n_critics must be 1..%d (got %d)", who, crit::MAX_CRITICS, n_critics);
    if (n_quantiles < 1 || n_quantiles > crit::MAX_QUANTILES || (kind == MVRL_CRITIC_SAC && n_quantiles != 1))
        return mvrl_fail(MVRL_EINVAL, "%s: n_quantiles must be 1..%d, and 1 for SAC (got %d)", who, crit::MAX_QUANTILES, n_quantiles);
    { const int rc = mvrl_require_device(device); if (rc != MVRL_OK) return rc; }
    MVRL_ON_DEVICE(device);
    MvrlCritic* h = new (std::nothrow) MvrlCritic();
    if (!h) return mvrl_fail(MVRL_EINVAL, "out of host memory");
    h->device = device; h->obs_dim = obs_dim; h->act_dim = act_dim; h->kind = kind; h->nc = n_critics; h->nq = n_quantiles;
    h->nqp = (n_quantiles + 15) / 16 * 16; h->packed = nullptr; h->has_weights = false;
    cudaError_t e = cudaMalloc(&h->packed, (size_t)n_critics * crit::critic_bytes(h->nqp));
    if (e == cudaSuccess) e = cudaFuncSetAttribute(crit::critic_target_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, crit::SMEM_BYTES);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(cgrad::critic_forward_kernel<cgrad::NET_CRITIC>, cudaFuncAttributeMaxDynamicSharedMemorySize, cgrad::FWD_SMEM_BYTES);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(cgrad::critic_backward_kernel<cgrad::NET_CRITIC>, cudaFuncAttributeMaxDynamicSharedMemorySize, cgrad::BWD_SMEM_BYTES);
    if (e != cudaSuccess) {
        if (h->packed) cudaFree(h->packed);
        delete h;
        return mvrl_fail(MVRL_ECUDA, "%s: %s", who, cudaGetErrorString(e));
    }
    *out = h;
    return MVRL_OK;
}

extern "C" MVRL_API int mvrl_critic_destroy(MvrlCritic* h) {
    if (!h) return MVRL_OK;
    { MvrlDeviceGuard guard(h->device); cudaFree(h->packed); }
    delete h;
    return MVRL_OK;
}

extern "C" MVRL_API int mvrl_critic_set_weights_device(MvrlCritic* h, const float* const* params, mvrl_stream_t stream) {
    static const char* const who = "mvrl_critic_set_weights_device";
    if (!h || !params) return mvrl_fail(MVRL_EINVAL, "%s: null argument", who);
    PackArgs p = {};
    for (int i = 0; i < 8 * h->nc; ++i) {
        if (!params[i]) return mvrl_fail(MVRL_EINVAL, "%s: null parameter %d (critic %d)", who, i, i / 8);
        p.cw[i] = params[i];
    }
    { const int rc = mvrl_check_device_ptrs(h->device, params, nullptr, 8 * h->nc, who); if (rc != MVRL_OK) return rc; }
    p.critic = reinterpret_cast<unsigned*>(h->packed);
    p.critic_words = h->nc * crit::critic_bytes(h->nqp) / 4;
    p.critic_k = h->obs_dim + h->act_dim; p.critic_nq = h->nq; p.critic_nqp = h->nqp;
    p.obs_dim = h->obs_dim; p.act_dim = h->act_dim;
    MVRL_ON_DEVICE(h->device);
    policy_pack_kernel<<<(p.critic_words + PACK_THREADS - 1) / PACK_THREADS, PACK_THREADS, 0, (cudaStream_t)stream>>>(p);
    const int rc = mvrl_check_launch("policy_pack (critic)");
    if (rc == MVRL_OK) h->has_weights = true;
    return rc;
}

extern "C" MVRL_API int mvrl_critic_target(MvrlCritic* h, const MvrlPolicy* actor, int64_t B, const float* next_obs, const float* rewards,
                                           const float* dones, const float* ent_coef, float gamma, int drop_per_net, uint64_t seed,
                                           int64_t* calls, float* target, float* next_actions, float* next_logp, float* eps,
                                           mvrl_stream_t stream) {
    static const char* const who = "mvrl_critic_target";
    if (!h || !actor || !next_obs || !rewards || !dones || !ent_coef || !calls || !target) return mvrl_fail(MVRL_EINVAL, "%s: null argument", who);
    if (actor->head != HEAD_SQUASHED || actor->precision != MVRL_POLICY_PRECISION_FP32 || actor->obs_dim != h->obs_dim ||
        actor->act_dim != h->act_dim || actor->device != h->device)
        return mvrl_fail(MVRL_EINVAL, "%s: the actor must be a squashed-head fp32 policy handle with obs_dim %d, act_dim %d on device %d",
                         who, h->obs_dim, h->act_dim, h->device);
    if (!actor->has_weights || !h->has_weights) return mvrl_fail(MVRL_EINVAL, "%s: the actor or the critics have no weights", who);
    if (B < 1 || B > INT32_MAX) return mvrl_fail(MVRL_EINVAL, "%s: B must be in [1, 2^31) (got %lld)", who, (long long)B);
    const int kept = h->nc * (h->nq - drop_per_net);
    if (drop_per_net < 0 || (h->kind == MVRL_CRITIC_SAC && drop_per_net != 0) || kept < 1)
        return mvrl_fail(MVRL_EINVAL, "%s: drop_per_net %d must be >= 0 (0 for SAC) and keep at least one of %d quantiles per critic",
                         who, drop_per_net, h->nq);
    const void* ptrs[] = {next_obs, rewards, dones, ent_coef, calls, target, next_actions, next_logp, eps};
    static const char* const names[] = {"next_obs", "rewards", "dones", "ent_coef", "calls", "target", "next_actions", "next_logp", "eps"};
    { const int rc = mvrl_check_device_ptrs(h->device, ptrs, names, 9, who); if (rc != MVRL_OK) return rc; }
    MVRL_ON_DEVICE(h->device);
    crit::CriticArgs a;
    a.actor = actor->packed5; a.critic = h->packed; a.n = B;
    a.next_obs = next_obs; a.rewards = rewards; a.dones = dones; a.ent_coef = ent_coef;
    a.gamma = gamma; a.logp_const = actor->logp_const;
    a.obs_dim = h->obs_dim; a.act_dim = h->act_dim; a.nc = h->nc; a.nq = h->nq; a.nqp = h->nqp;
    a.n_target = h->kind == MVRL_CRITIC_SAC ? 1 : kept;
    a.seed = seed; a.calls = reinterpret_cast<long long*>(calls);
    a.target = target; a.next_actions = next_actions; a.next_logp = next_logp; a.eps = eps;
    const unsigned grid = (unsigned)((B + TM - 1) / TM);
    crit::critic_target_kernel<<<grid, TM, crit::SMEM_BYTES, (cudaStream_t)stream>>>(a);
    return mvrl_check_launch("critic_target");
}

// ------------------------------------------------------------------------------------------- critics with gradients (K12)
static int check_critic_call(const MvrlCritic* h, int64_t B, const char* who) {
    if (!h) return mvrl_fail(MVRL_EINVAL, "%s: null handle", who);
    if (!h->has_weights) return mvrl_fail(MVRL_EINVAL, "%s: the critics have no weights (mvrl_critic_set_weights_device)", who);
    if (B < 1 || B > INT32_MAX) return mvrl_fail(MVRL_EINVAL, "%s: B must be in [1, 2^31) (got %lld)", who, (long long)B);
    return MVRL_OK;
}

extern "C" MVRL_API int64_t mvrl_critic_saved_bytes(const MvrlCritic* h, int64_t B) {
    if (!h || B < 1) return 0;
    return (int64_t)h->nc * 3 * ((B + TM - 1) / TM) * (H * TM) * (int64_t)sizeof(float);
}

extern "C" MVRL_API int64_t mvrl_critic_grad_scratch(const MvrlCritic* h, int64_t B) {
    if (!h || B < 1) return 0;
    const int64_t n_tiles = (B + TM - 1) / TM, tpc = cgrad::tiles_per_cta(n_tiles, h->nc), ctas = (n_tiles + tpc - 1) / tpc;
    return ((int64_t)h->nc * ctas * cgrad::part_floats(h->nqp) + (int64_t)h->nc * B * h->act_dim) * (int64_t)sizeof(float);
}

extern "C" MVRL_API int mvrl_critic_forward(MvrlCritic* h, int64_t B, const float* obs, const float* act, float* q, float* saved,
                                            mvrl_stream_t stream) {
    static const char* const who = "mvrl_critic_forward";
    { const int rc = check_critic_call(h, B, who); if (rc != MVRL_OK) return rc; }
    if (!obs || !act || !q) return mvrl_fail(MVRL_EINVAL, "%s: null argument", who);
    const void* ptrs[] = {obs, act, q, saved};
    static const char* const names[] = {"obs", "act", "q", "saved"};
    { const int rc = mvrl_check_device_ptrs(h->device, ptrs, names, 4, who); if (rc != MVRL_OK) return rc; }
    MVRL_ON_DEVICE(h->device);
    cgrad::FwdArgs a{};
    a.net = h->packed; a.n = B; a.n_tiles = (B + TM - 1) / TM;
    a.obs = obs; a.act = act; a.q = q; a.saved = saved;
    a.obs_dim = h->obs_dim; a.act_dim = h->act_dim; a.nc = h->nc; a.nq = h->nq; a.nqp = h->nqp;
    cgrad::critic_forward_kernel<cgrad::NET_CRITIC><<<dim3((unsigned)a.n_tiles, (unsigned)h->nc), TM, cgrad::FWD_SMEM_BYTES, (cudaStream_t)stream>>>(a);
    return mvrl_check_launch("critic_forward");
}

extern "C" MVRL_API int mvrl_critic_backward(MvrlCritic* h, int64_t B, const float* obs, const float* act, const float* saved,
                                             const float* grad_q, float* const* grads, float* grad_act, void* scratch,
                                             mvrl_stream_t stream) {
    static const char* const who = "mvrl_critic_backward";
    { const int rc = check_critic_call(h, B, who); if (rc != MVRL_OK) return rc; }
    if (!obs || !act || !saved || !grad_q || !scratch) return mvrl_fail(MVRL_EINVAL, "%s: null argument", who);
    if (!grads && !grad_act) return mvrl_fail(MVRL_EINVAL, "%s: nothing to compute (grads and grad_act are both null)", who);
    const void* ptrs[] = {obs, act, saved, grad_q, grad_act, scratch};
    static const char* const names[] = {"obs", "act", "saved", "grad_q", "grad_act", "scratch"};
    { const int rc = mvrl_check_device_ptrs(h->device, ptrs, names, 6, who); if (rc != MVRL_OK) return rc; }
    cgrad::ReduceArgs ra = {};
    if (grads) {
        for (int i = 0; i < 8 * h->nc; ++i) {
            if (!grads[i]) return mvrl_fail(MVRL_EINVAL, "%s: null gradient %d (critic %d)", who, i, i / 8);
            ra.grads[i] = grads[i];
        }
        const int rc = mvrl_check_device_ptrs(h->device, grads, nullptr, 8 * h->nc, who);
        if (rc != MVRL_OK) return rc;
    }
    MVRL_ON_DEVICE(h->device);
    const long n_tiles = (long)((B + TM - 1) / TM), tpc = cgrad::tiles_per_cta(n_tiles, h->nc), ctas = (n_tiles + tpc - 1) / tpc;
    float* part = static_cast<float*>(scratch);
    float* gact = part + (long)h->nc * ctas * cgrad::part_floats(h->nqp);
    cgrad::BwdArgs a{};
    a.net = h->packed; a.n = B; a.n_tiles = n_tiles; a.tpc = tpc;
    a.obs = obs; a.act = act; a.saved = saved; a.grad_q = grad_q;
    a.part = grads ? part : nullptr; a.gact = grad_act ? gact : nullptr;
    a.obs_dim = h->obs_dim; a.act_dim = h->act_dim; a.nc = h->nc; a.nq = h->nq; a.nqp = h->nqp;
    cgrad::critic_backward_kernel<cgrad::NET_CRITIC><<<dim3((unsigned)ctas, (unsigned)h->nc), TM, cgrad::BWD_SMEM_BYTES, (cudaStream_t)stream>>>(a);
    { const int rc = mvrl_check_launch("critic_backward"); if (rc != MVRL_OK) return rc; }
    ra.part = part; ra.gact = gact; ra.grad_act = grad_act; ra.n = B;
    ra.nc = h->nc; ra.nq = h->nq; ra.nqp = h->nqp; ra.k = h->obs_dim + h->act_dim; ra.act_dim = h->act_dim; ra.ctas = (int)ctas;
    const long words = (grads ? (long)h->nc * cgrad::part_floats(h->nqp) : 0) + (grad_act ? (long)B * h->act_dim : 0);
    cgrad::critic_grad_reduce_kernel<cgrad::NET_CRITIC><<<(unsigned)((words + cgrad::REDUCE_THREADS - 1) / cgrad::REDUCE_THREADS), cgrad::REDUCE_THREADS, 0,
                                       (cudaStream_t)stream>>>(ra);
    return mvrl_check_launch("critic_grad_reduce");
}

// --------------------------------------------------------------------------------------------- actor with gradients (K13)
static int check_actor_call(const MvrlPolicy* h, int64_t B, const char* who) {
    if (!h) return mvrl_fail(MVRL_EINVAL, "%s: null handle", who);
    if (h->head != HEAD_SQUASHED || h->precision != MVRL_POLICY_PRECISION_FP32)
        return mvrl_fail(MVRL_EINVAL, "%s: the handle must have the squashed head and the fp32 precision", who);
    if (!h->has_weights) return mvrl_fail(MVRL_EINVAL, "%s: the actor has no weights (mvrl_policy_set_weights_squashed_device)", who);
    if (B < 1 || B > INT32_MAX) return mvrl_fail(MVRL_EINVAL, "%s: B must be in [1, 2^31) (got %lld)", who, (long long)B);
    return MVRL_OK;
}
static bool is_actor(const MvrlPolicy* h) { return h && h->head == HEAD_SQUASHED && h->precision == MVRL_POLICY_PRECISION_FP32; }

extern "C" MVRL_API int64_t mvrl_actor_saved_bytes(const MvrlPolicy* h, int64_t B) {
    if (!is_actor(h) || B < 1) return 0;
    return (int64_t)cgrad::actor_saved_floats((B + TM - 1) / TM) * (int64_t)sizeof(float);
}

extern "C" MVRL_API int64_t mvrl_actor_grad_scratch(const MvrlPolicy* h, int64_t B) {
    if (!is_actor(h) || B < 1) return 0;
    const int64_t n_tiles = (B + TM - 1) / TM, tpc = cgrad::tiles_per_cta(n_tiles, 1), ctas = (n_tiles + tpc - 1) / tpc;
    return ctas * cgrad::part_floats(f32::HEAD_N) * (int64_t)sizeof(float);
}

extern "C" MVRL_API int mvrl_actor_forward(MvrlPolicy* h, int64_t B, const float* obs, float* actions, float* log_prob, float* eps,
                                           float* saved, uint64_t seed, int64_t* calls, mvrl_stream_t stream) {
    static const char* const who = "mvrl_actor_forward";
    { const int rc = check_actor_call(h, B, who); if (rc != MVRL_OK) return rc; }
    const void* ptrs[] = {obs, actions, log_prob, calls, eps, saved};
    static const char* const names[] = {"obs", "actions", "log_prob", "calls", "eps", "saved"};
    for (int i = 0; i < 4; ++i)
        if (!ptrs[i]) return mvrl_fail(MVRL_EINVAL, "%s: null argument %s", who, names[i]);
    { const int rc = mvrl_check_device_ptrs(h->device, ptrs, names, 6, who); if (rc != MVRL_OK) return rc; }
    MVRL_ON_DEVICE(h->device);
    cgrad::FwdArgs a{};
    a.net = h->packed5; a.n = B; a.n_tiles = (B + TM - 1) / TM;
    a.obs = obs; a.saved = saved;
    a.obs_dim = h->obs_dim; a.act_dim = h->act_dim; a.nc = 1; a.nqp = f32::HEAD_N;
    a.actions = actions; a.logp = log_prob; a.eps = eps; a.seed = seed; a.calls = reinterpret_cast<long long*>(calls);
    a.logp_const = h->logp_const;
    cgrad::critic_forward_kernel<cgrad::NET_ACTOR><<<(unsigned)a.n_tiles, TM, cgrad::FWD_SMEM_BYTES, (cudaStream_t)stream>>>(a);
    return mvrl_check_launch("actor_forward");
}

extern "C" MVRL_API int mvrl_actor_backward(MvrlPolicy* h, int64_t B, const float* obs, const float* saved, const float* grad_actions,
                                            const float* grad_log_prob, float* const* grads, void* scratch, mvrl_stream_t stream) {
    static const char* const who = "mvrl_actor_backward";
    static const char* const param_names[10] = {"latent_pi.0.weight", "latent_pi.0.bias", "latent_pi.2.weight", "latent_pi.2.bias",
                                                "latent_pi.4.weight", "latent_pi.4.bias", "mu.weight", "mu.bias", "log_std.weight",
                                                "log_std.bias"};
    { const int rc = check_actor_call(h, B, who); if (rc != MVRL_OK) return rc; }
    const void* ptrs[] = {obs, saved, grads, scratch, grad_actions, grad_log_prob};
    static const char* const names[] = {"obs", "saved", "grads", "scratch", "grad_actions", "grad_log_prob"};
    for (int i = 0; i < 4; ++i)
        if (!ptrs[i]) return mvrl_fail(MVRL_EINVAL, "%s: null argument %s", who, names[i]);
    if (!grad_actions && !grad_log_prob) return mvrl_fail(MVRL_EINVAL, "%s: nothing to differentiate (grad_actions and grad_log_prob are both null)", who);
    cgrad::ReduceArgs ra = {};
    for (int i = 0; i < 10; ++i) {
        if (!grads[i]) return mvrl_fail(MVRL_EINVAL, "%s: null gradient %s", who, param_names[i]);
        ra.grads[i] = grads[i];
    }
    const void* dptrs[] = {obs, saved, scratch, grad_actions, grad_log_prob};
    static const char* const dnames[] = {"obs", "saved", "scratch", "grad_actions", "grad_log_prob"};
    { const int rc = mvrl_check_device_ptrs(h->device, dptrs, dnames, 5, who); if (rc != MVRL_OK) return rc; }
    { const int rc = mvrl_check_device_ptrs(h->device, grads, param_names, 10, who); if (rc != MVRL_OK) return rc; }
    MVRL_ON_DEVICE(h->device);
    const long n_tiles = (long)((B + TM - 1) / TM), tpc = cgrad::tiles_per_cta(n_tiles, 1), ctas = (n_tiles + tpc - 1) / tpc;
    cgrad::BwdArgs a{};
    a.net = h->packed5; a.n = B; a.n_tiles = n_tiles; a.tpc = tpc;
    a.obs = obs; a.saved = saved; a.part = static_cast<float*>(scratch);
    a.obs_dim = h->obs_dim; a.act_dim = 0; a.nc = 1; a.nq = h->act_dim; a.nqp = f32::HEAD_N;
    a.grad_actions = grad_actions; a.grad_logp = grad_log_prob; a.head_dim = h->act_dim;
    cgrad::critic_backward_kernel<cgrad::NET_ACTOR><<<(unsigned)ctas, TM, cgrad::BWD_SMEM_BYTES, (cudaStream_t)stream>>>(a);
    { const int rc = mvrl_check_launch("actor_backward"); if (rc != MVRL_OK) return rc; }
    ra.part = a.part; ra.n = B; ra.nc = 1; ra.nq = h->act_dim; ra.nqp = f32::HEAD_N; ra.k = h->obs_dim; ra.ctas = (int)ctas;
    const long words = cgrad::part_floats(f32::HEAD_N);
    cgrad::critic_grad_reduce_kernel<cgrad::NET_ACTOR><<<(unsigned)((words + cgrad::REDUCE_THREADS - 1) / cgrad::REDUCE_THREADS),
                                                         cgrad::REDUCE_THREADS, 0, (cudaStream_t)stream>>>(ra);
    return mvrl_check_launch("actor_grad_reduce");
}
