// C ABI of the plain off-policy replay buffer (K9): SB3 2.x ReplayBuffer.add fed by OffPolicyAlgorithm._store_transition,
// and ReplayBuffer.sample / _get_samples, on the env's own feature-major buffers.  One launch per add, one per sample; the
// slot position and the sample-call counter live in a device cursor, so a CUDA graph of T adds / samples replayed R times
// behaves like T * R eager calls.
#include "mvrl_host.h"
#include "mvrl_math.cuh"

namespace mvrl {

constexpr int kAddEnvs = 128;      // environments per block of replay_add_kernel
constexpr int kAddThreads = 256;
constexpr int kSampleThreads = 256;
constexpr uint32_t kSampleStream = 9;   // Philox stream of the sampler (0: resets, 7 / 8: the actor's eps / action noise)

// One block stages its kAddEnvs environments' rows of one array in shared memory (feature-major reads, coalesced along the
// environments) and then stores the slot's contiguous run of cnt * k values (coalesced along the run).
template <typename T>
__device__ __forceinline__ void store_run(T* dst, const T* tile, int cnt, int k) {
    for (int j = threadIdx.x; j < cnt * k; j += blockDim.x) dst[j] = tile[j];
}

// cursor[0] = pos, [1] = adds, [2] = sample calls, [3] = pos << 32 | add blocks arrived, [4] = sample blocks arrived.
// Each add block takes pos and its ticket from cursor[3] in one atomicAdd; the block that draws the last ticket (every other
// block has already taken pos from the same word) alone advances pos (SB3: pos += 1; if pos == buffer_size: full, pos = 0),
// writes it back with the ticket count cleared, and publishes pos / adds in cursor[0] / [1] for the sampler and the host.
// Every access to cursor[3] within a launch is an atomic on one word, so no fence is needed.
template <typename T>
__global__ void __launch_bounds__(kAddThreads) replay_add_kernel(
        long n, long ld, int obs_dim, int act_dim, long slots, const T* __restrict__ obs, const T* __restrict__ terminal_obs,
        const T* __restrict__ act, const T* __restrict__ reward, const uint8_t* __restrict__ done, const uint8_t* __restrict__ timeout,
        T* __restrict__ last_obs, T* __restrict__ b_obs, T* __restrict__ b_next, T* __restrict__ b_act, T* __restrict__ b_rew,
        uint8_t* __restrict__ b_done, uint8_t* __restrict__ b_timeout, long long* cursor) {
    __shared__ T s_a[kAddEnvs * MVRL_REPLAY_MAX_DIM];
    __shared__ T s_b[kAddEnvs * MVRL_REPLAY_MAX_DIM];
    __shared__ long s_pos;
    if (threadIdx.x == 0) {
        const unsigned long long w = atomicAdd((unsigned long long*)&cursor[3], 1ull);
        s_pos = (long)(w >> 32);
        if ((unsigned)w == gridDim.x - 1) {
            const long next = s_pos + 1 == slots ? 0 : s_pos + 1;
            atomicExch((unsigned long long*)&cursor[3], (unsigned long long)next << 32);
            cursor[0] = next;
            cursor[1] += 1;
        }
    }
    __syncthreads();
    const long base = (long)blockIdx.x * kAddEnvs;
    const int cnt = (int)min((long)kAddEnvs, n - base);
    const long row0 = s_pos * n + base;   // first transition of this block in the slot
    // obs_t from the staging row (SB3's _last_obs), next_obs = terminal_obs where done else obs; the staging row is then
    // refreshed with the post-step obs (_last_obs = new_obs) - each element read and rewritten by the same thread
    for (int j = threadIdx.x; j < cnt * obs_dim; j += blockDim.x) {
        const int k = j / cnt, e = j - k * cnt;
        const long src = k * ld + base + e;
        const T o = obs[src];
        const T nx = (terminal_obs != nullptr && done[base + e]) ? terminal_obs[src] : o;
        s_a[e * obs_dim + k] = last_obs[src];
        s_b[e * obs_dim + k] = nx;
        last_obs[src] = o;
    }
    if (threadIdx.x < cnt) {
        const long i = base + threadIdx.x;
        b_rew[row0 + threadIdx.x] = reward[i];
        b_done[row0 + threadIdx.x] = done[i];
        b_timeout[row0 + threadIdx.x] = (timeout != nullptr && timeout[i] != 0) ? 1 : 0;
    }
    __syncthreads();
    store_run(b_obs + row0 * obs_dim, s_a, cnt, obs_dim);
    store_run(b_next + row0 * obs_dim, s_b, cnt, obs_dim);
    __syncthreads();
    for (int j = threadIdx.x; j < cnt * act_dim; j += blockDim.x) {
        const int k = j / cnt, e = j - k * cnt;
        s_a[e * act_dim + k] = act[k * ld + base + e];
    }
    __syncthreads();
    store_run(b_act + row0 * act_dim, s_a, cnt, act_dim);
}

// The sample call counter is 64-bit and cannot share a word with the ticket: device_call_number.
// One thread per sample.  slot = floor(u64 * size / 2^64), env = floor(u64' * n / 2^64) from one Philox4x32-10 block with
// counter (i, call_lo, call_hi, 9 * 65536) and key (seed_lo, seed_hi); size = slots if full else pos, as SB3's sample().
template <typename T>
__global__ void __launch_bounds__(kSampleThreads) replay_sample_kernel(
        long n, int obs_dim, int act_dim, long slots, long batch, uint64_t seed, const T* __restrict__ b_obs,
        const T* __restrict__ b_next, const T* __restrict__ b_act, const T* __restrict__ b_rew, const uint8_t* __restrict__ b_done,
        const uint8_t* __restrict__ b_timeout, long long* cursor, T* __restrict__ o_obs, T* __restrict__ o_act,
        T* __restrict__ o_next, T* __restrict__ o_done, T* __restrict__ o_rew) {
    __shared__ unsigned long long s_call;
    __shared__ long s_size;
    if (threadIdx.x == 0) {
        s_size = cursor[1] >= slots ? slots : (long)cursor[0];
        s_call = device_call_number(&cursor[2], &cursor[4]);
    }
    __syncthreads();
    const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= batch) return;
    const uint4 w = Philox::run(make_uint4((uint32_t)i, (uint32_t)s_call, (uint32_t)(s_call >> 32), kSampleStream * 65536u),
                                make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)));
    const long slot = (long)__umul64hi((uint64_t)w.x | ((uint64_t)w.y << 32), (uint64_t)s_size);
    const long env = (long)__umul64hi((uint64_t)w.z | ((uint64_t)w.w << 32), (uint64_t)n);
    const long row = slot * n + env;
    for (int k = 0; k < obs_dim; ++k) {
        o_obs[i * obs_dim + k] = b_obs[row * obs_dim + k];
        o_next[i * obs_dim + k] = b_next[row * obs_dim + k];
    }
    for (int k = 0; k < act_dim; ++k) o_act[i * act_dim + k] = b_act[row * act_dim + k];
    o_done[i] = T(b_done[row]) * (T(1) - T(b_timeout[row]));   // buffers.py: dones * (1 - timeouts)
    o_rew[i] = b_rew[row];
}

static int check_storage(const MvrlReplayStorage* s, int obs_dim, int act_dim, int64_t slots, const char* who) {
    if (!s || !s->observations || !s->next_observations || !s->actions || !s->rewards || !s->dones || !s->timeouts || !s->last_obs || !s->cursor)
        return mvrl_fail(MVRL_EINVAL, "%s: null storage pointer", who);
    if (obs_dim < 1 || obs_dim > MVRL_REPLAY_MAX_DIM || act_dim < 1 || act_dim > MVRL_REPLAY_MAX_DIM)
        return mvrl_fail(MVRL_EINVAL, "%s: obs_dim %d / act_dim %d outside [1, %d]", who, obs_dim, act_dim, MVRL_REPLAY_MAX_DIM);
    if (slots < 1) return mvrl_fail(MVRL_EINVAL, "%s: slots must be >= 1", who);
    return MVRL_OK;
}

}  // namespace mvrl

using namespace mvrl;

extern "C" MVRL_API int mvrl_replay_add(int dtype, int64_t n, int64_t ld, int obs_dim, int act_dim, int64_t slots,
                                        const MvrlReplayStorage* s, const void* obs, const void* terminal_obs, const void* act,
                                        const void* reward, const uint8_t* done, const uint8_t* timeout, mvrl_stream_t stream) {
    const char* who = "mvrl_replay_add";
    if (int rc = check_storage(s, obs_dim, act_dim, slots, who)) return rc;
    if (!obs || !act || !reward || !done) return mvrl_fail(MVRL_EINVAL, "%s: null argument", who);
    if (n < 1 || ld < n) return mvrl_fail(MVRL_EINVAL, "%s: need 1 <= n <= ld", who);
    if (dtype != MVRL_F32 && dtype != MVRL_F64) return mvrl_fail(MVRL_EINVAL, "%s: bad dtype", who);
    MVRL_ON_DEVICE_OF(s->observations, obs, who);
    const void* ptrs[] = {obs, s->next_observations, s->actions, s->rewards, s->dones, s->timeouts, s->last_obs, s->cursor,
                          terminal_obs, act, reward, done, timeout};
    static const char* const names[] = {"obs", "next_observations", "actions", "rewards", "dones", "timeouts", "last_obs", "cursor",
                                        "terminal_obs", "act", "reward", "done", "timeout"};
    if (int rc = mvrl_check_device_ptrs(mvrl_dev_out_, ptrs, names, 13, who)) return rc;
    const unsigned g = mvrl_grid_for(n, kAddEnvs);
    cudaStream_t st = (cudaStream_t)stream;
    long long* cur = (long long*)s->cursor;
    if (dtype == MVRL_F64)
        replay_add_kernel<double><<<g, kAddThreads, 0, st>>>(n, ld, obs_dim, act_dim, slots, (const double*)obs, (const double*)terminal_obs,
            (const double*)act, (const double*)reward, done, timeout, (double*)s->last_obs, (double*)s->observations,
            (double*)s->next_observations, (double*)s->actions, (double*)s->rewards, s->dones, s->timeouts, cur);
    else
        replay_add_kernel<float><<<g, kAddThreads, 0, st>>>(n, ld, obs_dim, act_dim, slots, (const float*)obs, (const float*)terminal_obs,
            (const float*)act, (const float*)reward, done, timeout, (float*)s->last_obs, (float*)s->observations,
            (float*)s->next_observations, (float*)s->actions, (float*)s->rewards, s->dones, s->timeouts, cur);
    return mvrl_check_launch("replay_add");
}

extern "C" MVRL_API int mvrl_replay_sample(int dtype, int64_t n, int obs_dim, int act_dim, int64_t slots, const MvrlReplayStorage* s,
                                           int64_t batch, uint64_t seed, void* out_obs, void* out_act, void* out_next_obs,
                                           void* out_dones, void* out_rewards, mvrl_stream_t stream) {
    const char* who = "mvrl_replay_sample";
    if (int rc = check_storage(s, obs_dim, act_dim, slots, who)) return rc;
    if (!out_obs || !out_act || !out_next_obs || !out_dones || !out_rewards) return mvrl_fail(MVRL_EINVAL, "%s: null output", who);
    if (n < 1) return mvrl_fail(MVRL_EINVAL, "%s: n must be >= 1", who);
    if (batch < 1 || batch > INT32_MAX) return mvrl_fail(MVRL_EINVAL, "%s: batch must be in [1, 2^31)", who);
    if (dtype != MVRL_F32 && dtype != MVRL_F64) return mvrl_fail(MVRL_EINVAL, "%s: bad dtype", who);
    MVRL_ON_DEVICE_OF(out_obs, s->observations, who);
    const void* ptrs[] = {s->observations, s->next_observations, s->actions, s->rewards, s->dones, s->timeouts, s->cursor,
                          out_act, out_next_obs, out_dones, out_rewards};
    static const char* const names[] = {"observations", "next_observations", "actions", "rewards", "dones", "timeouts", "cursor",
                                        "out_act", "out_next_obs", "out_dones", "out_rewards"};
    if (int rc = mvrl_check_device_ptrs(mvrl_dev_out_, ptrs, names, 11, who)) return rc;
    const unsigned g = mvrl_grid_for(batch, kSampleThreads);
    cudaStream_t st = (cudaStream_t)stream;
    long long* cur = (long long*)s->cursor;
    if (dtype == MVRL_F64)
        replay_sample_kernel<double><<<g, kSampleThreads, 0, st>>>(n, obs_dim, act_dim, slots, batch, seed, (const double*)s->observations,
            (const double*)s->next_observations, (const double*)s->actions, (const double*)s->rewards, s->dones, s->timeouts, cur,
            (double*)out_obs, (double*)out_act, (double*)out_next_obs, (double*)out_dones, (double*)out_rewards);
    else
        replay_sample_kernel<float><<<g, kSampleThreads, 0, st>>>(n, obs_dim, act_dim, slots, batch, seed, (const float*)s->observations,
            (const float*)s->next_observations, (const float*)s->actions, (const float*)s->rewards, s->dones, s->timeouts, cur,
            (float*)out_obs, (float*)out_act, (float*)out_next_obs, (float*)out_dones, (float*)out_rewards);
    return mvrl_check_launch("replay_sample");
}
