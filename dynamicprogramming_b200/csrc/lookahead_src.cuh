// lookahead_src.cuh — one-step lookahead on a value table: Q-values at any state and the controller that acts on them
// (NVRTC, sm_100a; DESIGN.md §8 N8, INTEGRATION.md §2e).
//
// Part of the rollout program: compile_rollout concatenates
//     [#define PI_D ...] + [#define PI_CALL_STEP_DYNAMICS ...] + [plugin source] + row_value_src.cuh + lookup_src.cuh
//     + rollout_src.cuh + this file
// and compiles it with the table builder's options, so step_dynamics is compiled from the same text under the same
// options as in the table builder.
//
// Definition.  V is a value table in reference order (n_states float32, the layout of a saved .npz) on the grid
// (lo, hi, shape) of g, with reference strides g.stride; gamma is float32.  For a query point x (D float32 values, not
// clamped or wrapped) and each action index a = 0 .. A-1:
//   1. step_dynamics(x, actions[a]) -> x', r, term (one call);
//   2. term: ev = 0.  Otherwise the table builder's cell search (table_build_src.h: pi_row) finds the cell of x':
//      n = (x' - lo) / (hi - lo) * (shape - 1), n = fmaxf(0, fminf(n, shape - 1)), i = min((int)n, shape - 2),
//      f = n - i; and ev = expected_value<D>(V, base, f, stride) (row_value_src.cuh): the reference's corner order and
//      its fmaf chain;
//   3. Q[a] = fmaf(gamma, ev, r);
//   4. the winner follows the improvement's rule: ascending a, strict '>' from -1e30f, starting at index 0.  The lowest
//      index wins ties, NaN never wins, and when nothing beats -1e30f the answer is action 0.
// The terminal mask is not consulted.  At a grid node that is not absorbing, with the V the improvement pass reads, the
// winner is the action pi_improve writes for that node, in both table modes and in every storage order: every
// floating-point operation after step_dynamics returns is an explicitly rounded intrinsic or an explicit fmaf, so the
// compiler cannot fuse a multiply of the plugin with the arithmetic here (the builder's own cell search is pinned to a
// contraction-free host restatement by tests/test_gpu_rollout.py).
#define PI_LOOKAHEAD_BLOCK 128

// Q-values of every action at x and the winner (the definition above).  q_out[a] = Q[a] when q_out is not null.
// Each action's step_dynamics call gets x through an opaque register move, so the compiler cannot hoist the part of the
// plugin that does not depend on the action out of the loop: every call is compiled as a single call with fresh inputs,
// as in pi_step_states and the table builder (a hoisted reward term was contracted differently on pendulum).
__device__ __forceinline__ int lookahead_point(const LookupGrid& g, const float (&x)[PI_D],
                                               const float* __restrict__ actions, const int n_actions,
                                               const float* __restrict__ V, const float gamma, float* __restrict__ q_out)
{
    int best = 0;
    float best_q = -1.0e30f;
    for (int a = 0; a < n_actions; ++a) {
        float pi_x[PI_D];
        #pragma unroll
        for (int d = 0; d < PI_D; ++d) asm volatile("mov.b32 %0, %1;" : "=f"(pi_x[d]) : "f"(x[d]));
        const float pi_action = actions[a];
        float pi_nx[PI_D];
        float pi_reward;
        bool pi_terminated;
        PI_CALL_STEP_DYNAMICS;

        float ev = 0.0f;
        if (!pi_terminated) {
            float frac[PI_D];
            int stride[PI_D];
            int base = 0;
            #pragma unroll
            for (int d = 0; d < PI_D; ++d) {
                const float top = (float)(g.shape[d] - 1);
                float n = __fmul_rn(__fdiv_rn(__fsub_rn(pi_nx[d], g.lo[d]), __fsub_rn(g.hi[d], g.lo[d])), top);
                n = fmaxf(0.0f, fminf(n, top));
                const int i = min((int)n, g.shape[d] - 2);
                frac[d] = __fsub_rn(n, (float)i);
                stride[d] = g.stride[d];
                base += i * g.stride[d];
            }
            ev = expected_value<PI_D>(V, base, frac, stride);
        }
        const float q = fmaf(gamma, ev, pi_reward);
        if (q_out != nullptr) q_out[a] = q;
        if (q > best_q) { best_q = q; best = a; }
    }
    return best;
}

// One thread per query point: the winner's index (best_action, may be null) and the n x A row-major Q matrix (q, may be
// null).
extern "C" __global__ void __launch_bounds__(PI_LOOKAHEAD_BLOCK)
pi_lookahead_points(const LookupGrid g, const float* __restrict__ actions, const int n_actions,
                    const float* __restrict__ V, const float gamma, const float* __restrict__ points, const long long n,
                    int* __restrict__ best_action, float* __restrict__ q)
{
    const long long i = (long long)blockIdx.x * PI_LOOKAHEAD_BLOCK + threadIdx.x;
    if (i >= n) return;
    float pi_x[PI_D];
    #pragma unroll
    for (int d = 0; d < PI_D; ++d) pi_x[d] = points[i * PI_D + d];
    const int a = lookahead_point(g, pi_x, actions, n_actions, V, gamma, q != nullptr ? q + i * n_actions : nullptr);
    if (best_action != nullptr) best_action[i] = a;
}

// pi_rollout_episodes with the lookahead as the controller: a_t = lookahead_point(x_t) with Q under gamma_q =
// (float)gamma, then the step, the float64 return sums (discounted with gamma) and the recording layout of
// pi_rollout_episodes; the recorded action is actions[a_t].
extern "C" __global__ void __launch_bounds__(PI_ROLLOUT_BLOCK)
pi_rollout_lookahead(const LookupGrid g, const float* __restrict__ actions, const int n_actions,
                     const float* __restrict__ V, const float gamma_q,
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
        const float pi_action = actions[lookahead_point(g, pi_x, actions, n_actions, V, gamma_q, nullptr)];
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
