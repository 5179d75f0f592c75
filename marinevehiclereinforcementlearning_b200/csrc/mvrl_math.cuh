// Small device-side math layer shared by every kernel of libmvrl.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <math.h>

// Rare paths (libm fmod, Philox resets) are __noinline__ so that they do not bloat the instruction stream every warp
// fetches.

namespace mvrl {

// ---- precision-generic libm wrappers -------------------------------------
template <typename T> struct Real;
template <> struct Real<float> {
    static __device__ __forceinline__ void sincos(float x, float* s, float* c) { sincosf(x, s, c); }
    static __device__ __forceinline__ float sqrt(float x) { return sqrtf(x); }
    static __device__ __forceinline__ float exp(float x) { return expf(x); }
    static __device__ __forceinline__ float fmod(float a, float b) { return fmodf(a, b); }
    static __device__ __forceinline__ float floor(float a) { return floorf(a); }
    static __device__ __forceinline__ float nan() { return __int_as_float(0x7fc00000); }
};
template <> struct Real<double> {
    static __device__ __forceinline__ void sincos(double x, double* s, double* c) { ::sincos(x, s, c); }
    static __device__ __forceinline__ double sqrt(double x) { return ::sqrt(x); }
    static __device__ __forceinline__ double exp(double x) { return ::exp(x); }
    static __device__ __forceinline__ double fmod(double a, double b) { return ::fmod(a, b); }
    static __device__ __forceinline__ double floor(double a) { return ::floor(a); }
    static __device__ __forceinline__ double nan() { return __longlong_as_double(0x7ff8000000000000LL); }
};

template <typename T> __device__ __forceinline__ T tabs(T x) { return x < T(0) ? -x : x; }
template <> __device__ __forceinline__ float tabs<float>(float x) { return fabsf(x); }
template <> __device__ __forceinline__ double tabs<double>(double x) { return fabs(x); }
__device__ __forceinline__ float fmaf_t(float a, float b, float c) { return fmaf(a, b, c); }
__device__ __forceinline__ double fmaf_t(double a, double b, double c) { return fma(a, b, c); }
template <typename T> __device__ __forceinline__ T tmin(T a, T b) { return a < b ? a : b; }
template <typename T> __device__ __forceinline__ T tmax(T a, T b) { return a > b ? a : b; }
template <typename T> __device__ __forceinline__ T clampt(T x, T lo, T hi) { return tmax(lo, tmin(hi, x)); }
// numpy.sign: -1, 0, +1
template <typename T> __device__ __forceinline__ T sgn(T x) { return x > T(0) ? T(1) : (x < T(0) ? T(-1) : T(0)); }
template <typename T> __device__ __forceinline__ bool finite_t(T x);
template <> __device__ __forceinline__ bool finite_t<double>(double x) { return isfinite(x); }
template <> __device__ __forceinline__ bool finite_t<float>(float x) { return isfinite(x); }

// ---- value types ----------------------------------------------------------
// The model code is written once over a value type V: float / double carry one
// environment per thread; F2 carries TWO fp32 environments per thread in a
// register pair and maps +, *, fma onto the packed FFMA2 / FADD2 / FMUL2
// instructions of sm_100 (two FMAs per lane per issue slot; scalar and uniform
// operands broadcast for free, neg / abs are operand modifiers).  The step
// kernels are issue-bound, not pipe-bound, so halving the issue slots of the
// FP work is a direct speed-up (profiles/ r1 notes).
struct F2 {
    float2 v;
    __device__ __forceinline__ F2() {}
    __device__ __forceinline__ F2(float a) { v = make_float2(a, a); }
    __device__ __forceinline__ F2(float a, float b) { v = make_float2(a, b); }
};
__device__ __forceinline__ F2 f2_from(float2 q) { F2 r; r.v = q; return r; }
__device__ __forceinline__ F2 operator-(F2 a) { return F2(-a.v.x, -a.v.y); }
__device__ __forceinline__ F2 operator+(F2 a, F2 b) { return f2_from(__fadd2_rn(a.v, b.v)); }
__device__ __forceinline__ F2 operator-(F2 a, F2 b) { return f2_from(__fadd2_rn(a.v, (-b).v)); }
__device__ __forceinline__ F2 operator*(F2 a, F2 b) { return f2_from(__fmul2_rn(a.v, b.v)); }
__device__ __forceinline__ F2& operator+=(F2& a, F2 b) { a = a + b; return a; }
__device__ __forceinline__ F2 fmaf_t(F2 a, F2 b, F2 c) { return f2_from(__ffma2_rn(a.v, b.v, c.v)); }
__device__ __forceinline__ F2 tabs(F2 a) { return F2(fabsf(a.v.x), fabsf(a.v.y)); }
__device__ __forceinline__ F2 tmin(F2 a, F2 b) { return F2(fminf(a.v.x, b.v.x), fminf(a.v.y, b.v.y)); }
__device__ __forceinline__ F2 tmax(F2 a, F2 b) { return F2(fmaxf(a.v.x, b.v.x), fmaxf(a.v.y, b.v.y)); }

template <typename V> struct VT { using S = V; static constexpr int L = 1; };
template <> struct VT<F2> { using S = float; static constexpr int L = 2; };

// lane access (l is a compile-time constant after unrolling)
template <typename V> __device__ __forceinline__ V lane_get(V v, int) { return v; }
__device__ __forceinline__ float lane_get(F2 v, int l) { return l == 0 ? v.v.x : v.v.y; }
template <typename V> __device__ __forceinline__ void lane_set(V& v, int, V x) { v = x; }
__device__ __forceinline__ void lane_set(F2& v, int l, float x) { if (l == 0) v.v.x = x; else v.v.y = x; }

// comparisons / selects: bool for one environment, a pair of predicates for two
struct B2 { bool x, y; };
template <typename T> __device__ __forceinline__ bool vlt(T a, T b) { return a < b; }
__device__ __forceinline__ B2 vlt(F2 a, F2 b) { return B2{a.v.x < b.v.x, a.v.y < b.v.y}; }
template <typename T> __device__ __forceinline__ bool vgt(T a, T b) { return a > b; }
__device__ __forceinline__ B2 vgt(F2 a, F2 b) { return B2{a.v.x > b.v.x, a.v.y > b.v.y}; }
template <typename T> __device__ __forceinline__ bool visnan(T a) { return a != a; }
__device__ __forceinline__ B2 visnan(F2 a) { return B2{a.v.x != a.v.x, a.v.y != a.v.y}; }
template <typename T> __device__ __forceinline__ T vsel(bool m, T a, T b) { return m ? a : b; }
__device__ __forceinline__ F2 vsel(B2 m, F2 a, F2 b) { return F2(m.x ? a.v.x : b.v.x, m.y ? a.v.y : b.v.y); }
// 1.0 / 0.0 masks for multiplicative selects: ONE instruction per lane (FSET.BF) where compare + select takes two, and the
// multiply that applies them is a packed FMA-pipe instruction - the set-point kernel was bound by the ALU pipe (profiles/
// r1_x: pipe_alu 40 % of issue slots against pipe_fma 32 %), so selects of the form "x or 0" are written mask * x.
template <typename T> __device__ __forceinline__ T vmask_lt(T a, T b) { return a < b ? T(1) : T(0); }
template <typename T> __device__ __forceinline__ T vmask_ge(T a, T b) { return a >= b ? T(1) : T(0); }
template <typename T> __device__ __forceinline__ T vmask_le(T a, T b) { return a <= b ? T(1) : T(0); }
__device__ __forceinline__ F2 vmask_lt(F2 a, F2 b) { return F2(a.v.x < b.v.x ? 1.0f : 0.0f, a.v.y < b.v.y ? 1.0f : 0.0f); }
__device__ __forceinline__ F2 vmask_ge(F2 a, F2 b) { return F2(a.v.x >= b.v.x ? 1.0f : 0.0f, a.v.y >= b.v.y ? 1.0f : 0.0f); }
__device__ __forceinline__ F2 vmask_le(F2 a, F2 b) { return F2(a.v.x <= b.v.x ? 1.0f : 0.0f, a.v.y <= b.v.y ? 1.0f : 0.0f); }
template <typename T> __device__ __forceinline__ bool vge(T a, T b) { return a >= b; }
__device__ __forceinline__ B2 vge(F2 a, F2 b) { return B2{a.v.x >= b.v.x, a.v.y >= b.v.y}; }
__device__ __forceinline__ bool vany(bool m) { return m; }
__device__ __forceinline__ bool vany(B2 m) { return m.x || m.y; }
__device__ __forceinline__ float vcopysign(float mag, float sign) { return copysignf(mag, sign); }
__device__ __forceinline__ double vcopysign(double mag, double sign) { return copysign(mag, sign); }
__device__ __forceinline__ F2 vcopysign(F2 mag, F2 sign) { return F2(copysignf(mag.v.x, sign.v.x), copysignf(mag.v.y, sign.v.y)); }

#define MVRL_TWO_PI 6.283185307179586476925286766559

// Python's float `%` (== numpy.mod): result takes the divisor's sign, and an
// exact zero remainder is +0 for a positive divisor.  The reference wraps
// angles with it (dynamicsModel_BlueROV2_Heavy_6DoF.py:560, resources.py:92-93).
// -b < a < 2b (the overwhelmingly common case: an angle wrapped one step ago, moved by less than a turn):
// no fmod, no branch.  a - b is exact for b <= a < 2b (Sterbenz), which is what fmod returns there.
template <typename T> __device__ __forceinline__ T pymod_small(T a, T b) { return a < T(0) ? a + b : (a >= b ? a - b : tabs(a)); }
// the same value from one add of a selected shift: a + 0 == |a| on [0, b) and turns -0 into +0 like the reference's %.  Straight-line
// code for the 6DoF step kernel's two-environment epilogue (+0.6 %); the legacy step kernel is 21 % SLOWER with it (the compiler
// schedules its loads differently around the selects, measured r1_auvab), so it keeps the form above.
template <typename T> __device__ __forceinline__ T pymod_small_sel(T a, T b) {
    const T shift = a < T(0) ? b : (a >= b ? -b : T(0));
    return a + shift;
}
// general case, kept out of line: libm's fmod carries a long slow path that would otherwise be
// inlined at every call site of the step kernels (measured: instruction-fetch stalls in the epilogue)
template <typename T> __device__ __noinline__ T pymod_general(T a, T b) {
    T r = Real<T>::fmod(a, b);
    if (r != T(0)) { if (r < T(0)) r += b; }
    else r = T(0);
    return r;
}
template <typename T> __device__ __forceinline__ T pymod_pos(T a, T b) {  // b > 0
    if (a > -b && a < b + b) return pymod_small(a, b);
    return pymod_general(a, b);
}

// resources.angleError (resources.py:75-95): a = (psi_d - psi) % 2pi, b = (psi - psi_d) % 2pi, a if a < b else -b
template <typename T> __device__ __forceinline__ T angle_error_small(T d) {   // d = psi_d - psi, |d| < 2 pi
    const T tp = T(MVRL_TWO_PI);
    const T a = d < T(0) ? d + tp : tabs(d), b = d > T(0) ? tp - d : tabs(d);   // d % 2pi and (-d) % 2pi for |d| < 2pi
    return a < b ? a : -b;
}
template <typename T> __device__ __forceinline__ T angle_error(T psi_d, T psi) {
    const T tp = T(MVRL_TWO_PI);
    const T d = psi_d - psi;                 // psi - psi_d == -d exactly
    if (tabs(d) < tp) return angle_error_small(d);
    const T a = pymod_general(d, tp), b = pymod_general(-d, tp);
    return a < b ? a : -b;
}

__device__ __forceinline__ F2 angle_error(F2 psi_d, F2 psi) {
    return F2(angle_error(psi_d.v.x, psi.v.x), angle_error(psi_d.v.y, psi.v.y));
}
// The same function, straight-line for any value type.  For |d| < 2 pi the selection of resources.py:92-95 (a = d % 2pi,
// b = -d % 2pi, a if a < b else -b) is d shifted by one turn when it lies outside [-pi, pi): a < b <=> d < -pi for
// negative d (result d + 2pi) and a >= b <=> d >= pi for positive d (result d - 2pi); both sums are exact where they
// apply (Sterbenz), so the value is the reference's bit for bit - except that equal angles give +0 where the reference
// gives -0.0.  Anything beyond one turn takes the exact out-of-line path.
#define MVRL_PI 3.141592653589793238462643383279
template <typename T> __device__ __noinline__ T angle_error_general(T psi_d, T psi) { return angle_error(psi_d, psi); }
__device__ __forceinline__ F2 angle_error_general(F2 psi_d, F2 psi) {
    return F2(angle_error_general(psi_d.v.x, psi.v.x), angle_error_general(psi_d.v.y, psi.v.y));
}
template <typename V> __device__ __forceinline__ V angle_error_v(V psi_d, V psi) {
    using S = typename VT<V>::S;
    const V d = psi_d - psi;
    const V turns = vmask_lt(d, V(S(-MVRL_PI))) - vmask_ge(d, V(S(MVRL_PI)));
    V e = fmaf_t(V(S(MVRL_TWO_PI)), turns, d);
    if (vany(vge(tabs(d), V(S(MVRL_TWO_PI))))) e = angle_error_general(psi_d, psi);
    return e;
}

// y += inc with a Kahan carry (compensated summation across RK4 sub-steps)
template <typename T> __device__ __forceinline__ void rk4_pose_update(T& y, T& carry, T inc) {
    const T t = inc - carry;
    const T s = y + t;
    carry = (s - y) - t;
    y = s;
}

__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }

// ---- Philox4x32-10 ---------------------------------------------------------
struct Philox {
    static __device__ __forceinline__ uint4 run(uint4 c, uint2 k) {
#pragma unroll
        for (int i = 0; i < 10; ++i) {
            uint32_t hi0 = __umulhi(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
            uint32_t hi1 = __umulhi(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
            c = make_uint4(hi1 ^ c.y ^ k.x, lo1, hi0 ^ c.w ^ k.y, lo0);
            k.x += 0x9E3779B9u; k.y += 0xBB67AE85u;
        }
        return c;
    }
    // block `blk` of the draw stream of (env, episode)
    static __device__ __forceinline__ uint4 draw(uint64_t seed, uint64_t env, uint32_t episode, uint32_t stream, uint32_t blk) {
        return run(make_uint4((uint32_t)env, (uint32_t)(env >> 32), episode, stream * 65536u + blk),
                   make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)));
    }
};
// The 64-bit call number of a launch, by thread 0 of each block: read *call, fence, take a ticket from *ticket; the block
// that draws the last ticket has seen every block's read and alone advances *call and clears *ticket (0 between launches).
// No host value is involved, so a CUDA graph of the launch replayed R times counts like R eager launches.
__device__ __forceinline__ unsigned long long device_call_number(long long* call, long long* ticket) {
    const unsigned long long c = (unsigned long long)*call;
    __threadfence();
    if (atomicAdd((unsigned long long*)ticket, 1ull) == gridDim.x - 1) {
        __threadfence();
        *call = (long long)(c + 1);
        *ticket = 0;
    }
    return c;
}
// 24-bit uniform in [0,1): exact in fp32 and fp64
template <typename T> __device__ __forceinline__ T u01(uint32_t w) { return T(w >> 8) * T(1.0 / 16777216.0); }

// ---- warp helpers ----------------------------------------------------------
__device__ __forceinline__ double warp_sum(double v, unsigned mask) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(mask, v, o);
    return v;
}
__device__ __forceinline__ double warp_min(double v, unsigned mask) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmin(v, __shfl_xor_sync(mask, v, o));
    return v;
}
__device__ __forceinline__ double warp_max(double v, unsigned mask) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(mask, v, o));
    return v;
}
// min / max of a double in global memory without a read-compare-swap loop: IEEE doubles order like signed
// integers when non-negative and like reversed unsigned integers when negative, so one integer atomic of the
// right flavour does it - and since the result is not used it is a fire-and-forget RED, no round trip to L2
// (the CAS loop's leading load was 12 % of the legacy step kernel's stall samples, profiles/ r1t).  NaN is
// never passed (non-finite environments are counted separately).
__device__ __forceinline__ void atomic_min_double(double* addr, double v) {
    v += 0.0;   // -0.0 -> +0.0: its bit pattern would otherwise compare as the most negative integer
    if (v >= 0.0) atomicMin((long long*)addr, __double_as_longlong(v));
    else atomicMax((unsigned long long*)addr, (unsigned long long)__double_as_longlong(v));
}
__device__ __forceinline__ void atomic_max_double(double* addr, double v) {
    v += 0.0;
    if (v >= 0.0) atomicMax((long long*)addr, __double_as_longlong(v));
    else atomicMin((unsigned long long*)addr, (unsigned long long)__double_as_longlong(v));
}

}  // namespace mvrl
