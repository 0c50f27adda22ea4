// rollout_src.cuh — closed-loop policy rollouts simulated with the plugin's own dynamics (NVRTC, sm_100a).
//
// What the reference's evaluate() does one step at a time on the CPU — get_optimal_action (utils/barycentric.py:76-108)
// followed by an environment step (e.g. runners/pendulum_cuda.py:161-166) — for a whole batch of episodes at once.
// The engine concatenates
//     [#define PI_D ...] + [#define PI_CALL_STEP_DYNAMICS ...] + [plugin source] + lookup_src.cuh + this file
// and compiles it with the table builder's options (architecture only: fmad on, IEEE division, like cupy.RawModule),
// so step_dynamics is compiled from the same text under the same options as in the table builder.
//
// Contraction: every value step_dynamics returns is used only by plain stores, by the explicitly rounded intrinsics of
// lookup_point and of the float64 return sums, and as an input of the next step_dynamics call.  Each next-state
// component has several uses (lookup, next step, optional record), so no multiply of the plugin can be fused with an
// operation of the caller: x_{t+1} and r_t are the values the plugin computes, as pi_step_states returns them.
#define PI_ROLLOUT_BLOCK 64
#define PI_STEP_BLOCK 256

// One thread runs one whole episode; the state stays in registers.  For t = 0..n_steps-1 until step_dynamics sets
// *terminated: a_t = lookup(x_t); step; total += r_t; ret += disc * r_t; disc *= gamma (float64, explicitly rounded).
// Recorded values are staged step-major (row t*D + d of a rows x n matrix; lanes of a warp store neighbouring words);
// pi_kernels.cuh: rollout_unstage_kernel turns them into the episode-major host layout.
extern "C" __global__ void __launch_bounds__(PI_ROLLOUT_BLOCK)
pi_rollout_episodes(const LookupGrid g, const int* __restrict__ policy, const float* __restrict__ actions,
                    const float* __restrict__ x0, const long long n, const int n_steps, const double gamma,
                    double* __restrict__ total_reward, double* __restrict__ discounted_return, int* __restrict__ length,
                    unsigned char* __restrict__ terminated, float* __restrict__ final_states,
                    float* __restrict__ rec_states, float* __restrict__ rec_actions, float* __restrict__ rec_rewards)
{
    const long long e = (long long)blockIdx.x * PI_ROLLOUT_BLOCK + threadIdx.x;
    if (e >= n) return;
    const bool rec = rec_states != nullptr;
    float pi_x[PI_D];
    #pragma unroll
    for (int d = 0; d < PI_D; ++d) pi_x[d] = x0[e * PI_D + d];
    if (rec) {
        #pragma unroll
        for (int d = 0; d < PI_D; ++d) rec_states[(long long)d * n + e] = pi_x[d];
    }
    double total = 0.0, ret = 0.0, disc = 1.0;
    int len = 0;
    bool done = false;
    for (int t = 0; t < n_steps && !done; ++t) {
        const float pi_action = lookup_point(g, PI_D, pi_x, policy, actions);
        float pi_nx[PI_D];
        float pi_reward;
        bool pi_terminated;
        PI_CALL_STEP_DYNAMICS;

        const double r = (double)pi_reward;
        total = __dadd_rn(total, r);
        ret = __dadd_rn(ret, __dmul_rn(disc, r));
        disc = __dmul_rn(disc, gamma);
        len = t + 1;
        done = pi_terminated;
        #pragma unroll
        for (int d = 0; d < PI_D; ++d) pi_x[d] = pi_nx[d];
        if (rec) {
            const long long row = (long long)(t + 1) * PI_D;
            #pragma unroll
            for (int d = 0; d < PI_D; ++d) rec_states[(row + d) * n + e] = pi_x[d];
            rec_actions[(long long)t * n + e] = pi_action;
            rec_rewards[(long long)t * n + e] = pi_reward;
        }
    }
    total_reward[e] = total;
    discounted_return[e] = ret;
    length[e] = len;
    terminated[e] = done ? 1 : 0;
    #pragma unroll
    for (int d = 0; d < PI_D; ++d) final_states[e * PI_D + d] = pi_x[d];
}

// One thread per (state, action) pair: a single step_dynamics call, outputs stored as they are.
extern "C" __global__ void __launch_bounds__(PI_STEP_BLOCK)
pi_step_states(const float* __restrict__ states, const float* __restrict__ acts, const long long n,
               float* __restrict__ next_states, float* __restrict__ rewards, unsigned char* __restrict__ terminated)
{
    const long long i = (long long)blockIdx.x * PI_STEP_BLOCK + threadIdx.x;
    if (i >= n) return;
    float pi_x[PI_D];
    #pragma unroll
    for (int d = 0; d < PI_D; ++d) pi_x[d] = states[i * PI_D + d];
    const float pi_action = acts[i];
    float pi_nx[PI_D];
    float pi_reward;
    bool pi_terminated;
    PI_CALL_STEP_DYNAMICS;
    #pragma unroll
    for (int d = 0; d < PI_D; ++d) next_states[i * PI_D + d] = pi_nx[d];
    rewards[i] = pi_reward;
    terminated[i] = pi_terminated ? 1 : 0;
}
