// table_build_src.h — CUDA source of the transition-table builder.
//
// This is the ONE kernel that has to be compiled at run time, because the
// environment plugin hands the engine its dynamics as a CUDA source string
// (`_dynamics_cuda_src()`, src/cuda_policy_iteration.py:113-125, :518-530,
// :941-954).  The engine concatenates
//     [#define PI_D ...] + [plugin source] + [kTableBuildSrc]
// and compiles it with NVRTC for sm_100a with default options (fmad on, IEEE
// division, no fast-math — what cupy.RawModule does at :289), so the compiler
// sees the plugin's expressions exactly as it does in the reference kernels.
//
// One thread per (state, action): decode the flat state index into grid
// coordinates, read the node coordinates from the per-axis arrays (the same
// float32 bits as the reference's states_space rows), run step_dynamics, apply
// the multilinear cell search of get_barycentric_{2,4,6}d
// (src/cuda_policy_iteration.py:183-199, :586-598, :1013-1027) and write one
// compact row with 128-bit coalesced stores.
//
// The same program holds the recompute-mode kernels (DESIGN.md §8 N7): pi_improve_recompute and pi_policy_rows get
// their rows from pi_row, the builder's own row function, and share expected_value / count_regular_groups with the
// ahead-of-time kernels (row_value_src.cuh, prepended by compile_to_cubin).  pi_build_rows keeps its store sequence
// inline rather than calling pi_store_row: that way its SASS stays what it was before these kernels were added.
#pragma once

namespace pi {

static const char* const kTableBuildSrc = R"PISRC(

typedef unsigned long long pi_size;
#define PI_W (PI_D + 2)
#define PI_N4 (PI_W / 4)
#define PI_N2 ((PI_W % 4) / 2)
#define PI_N1 (PI_W % 2)

struct PiBuildParams {
    unsigned char* table;          // [A] row tables (plane-SoA), action stride PI_W*4*n_pad bytes
    const float* actions;          // n_actions
    const unsigned char* absorbing; // local terminal mask (n_local), may be null
    const float* axes[PI_D];       // node coordinates per dimension
    long long n_local;
    long long n_pad;
    long long s_begin;             // first global state of this shard
    int n_actions;
    int shape[PI_D];
    int stride[PI_D];              // INTERNAL storage strides, indexed by logical dimension
    float lo[PI_D];
    float hi[PI_D];
    int perm[PI_D];                // storage position (0 = slowest) -> logical dimension
};

__device__ __forceinline__ void pi_st16(void* p, unsigned a, unsigned b, unsigned c, unsigned d) {
    asm volatile("st.global.L1::no_allocate.v4.u32 [%0], {%1,%2,%3,%4};" :: "l"(p), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}
__device__ __forceinline__ void pi_st8(void* p, unsigned a, unsigned b) {
    asm volatile("st.global.L1::no_allocate.v2.u32 [%0], {%1,%2};" :: "l"(p), "r"(a), "r"(b) : "memory");
}
__device__ __forceinline__ void pi_st4(void* p, unsigned a) {
    asm volatile("st.global.L1::no_allocate.u32 [%0], %1;" :: "l"(p), "r"(a) : "memory");
}

// The row of (local state pi_s, action index pi_a): node decode, the plugin's step_dynamics, the cell search and the
// sentinels.  Every kernel of this program that needs a row calls this one function with one (state, action) per
// thread and the action value read from p.actions, so step_dynamics is compiled in the same surroundings everywhere
// (DESIGN.md §3: the compiler's contraction choices depend on the code around the call).
__device__ __forceinline__ void pi_row(const PiBuildParams& p, const long long pi_s, const int pi_a, unsigned (&pi_w)[PI_W])
{
    #pragma unroll
    for (int k = 0; k < PI_W; ++k) pi_w[k] = 0u;

    if (p.absorbing != nullptr && p.absorbing[pi_s]) {
        pi_w[0] = (unsigned)(-2);                       // PI_ROW_ABSORBING
    } else {
        // internal flat index -> node coordinates (storage position k holds dimension perm[k])
        float pi_x[PI_D];
        unsigned pi_r = (unsigned)(p.s_begin + pi_s);
        #pragma unroll
        for (int k = PI_D - 1; k >= 0; --k) {
            const int pi_d = p.perm[k];
            const unsigned pi_q = pi_r / (unsigned)p.shape[pi_d];
            const unsigned pi_i = pi_r - pi_q * (unsigned)p.shape[pi_d];
            #pragma unroll
            for (int d = 0; d < PI_D; ++d)
                if (d == pi_d) pi_x[d] = p.axes[d][pi_i];
            pi_r = pi_q;
        }
        const float pi_action = p.actions[pi_a];
        float pi_nx[PI_D];
        float pi_reward;
        bool pi_terminated;
        PI_CALL_STEP_DYNAMICS;

        pi_w[PI_D + 1] = __float_as_uint(pi_reward);
        if (pi_terminated) {
            pi_w[0] = (unsigned)(-1);                   // PI_ROW_TERMINATED: sum_c w_c V_c := 0
        } else {
            int pi_base = 0;
            #pragma unroll
            for (int d = 0; d < PI_D; ++d) {
                // get_barycentric_Nd: normalise, clamp, truncate, fractional part
                float pi_n = (pi_nx[d] - p.lo[d]) / (p.hi[d] - p.lo[d]) * (float)(p.shape[d] - 1);
                pi_n = fmaxf(0.0f, fminf(pi_n, (float)(p.shape[d] - 1)));
                const int pi_i = min((int)pi_n, p.shape[d] - 2);
                const float pi_f = pi_n - (float)pi_i;
                pi_base += pi_i * p.stride[d];
                pi_w[1 + d] = __float_as_uint(pi_f);
            }
            pi_w[0] = (unsigned)pi_base;
        }
    }
}

// Store the row of local state pi_s into the plane-SoA table at pi_t (n_pad states per plane).
__device__ __forceinline__ void pi_store_row(unsigned char* pi_t, const long long n_pad, const long long pi_s, const unsigned (&pi_w)[PI_W])
{
    #pragma unroll
    for (int k = 0; k < PI_N4; ++k)
        pi_st16(pi_t + (pi_size)k * 16u * (pi_size)n_pad + (pi_size)pi_s * 16u,
                pi_w[4 * k], pi_w[4 * k + 1], pi_w[4 * k + 2], pi_w[4 * k + 3]);
#if (PI_W % 4) >= 2
    pi_st8(pi_t + (pi_size)PI_N4 * 16u * (pi_size)n_pad + (pi_size)pi_s * 8u,
           pi_w[4 * PI_N4], pi_w[4 * PI_N4 + 1]);
#endif
#if (PI_W % 2) == 1
    pi_st4(pi_t + ((pi_size)PI_N4 * 16u + (pi_size)PI_N2 * 8u) * (pi_size)n_pad + (pi_size)pi_s * 4u,
           pi_w[PI_W - 1]);
#endif
}

extern "C" __global__ void __launch_bounds__(256) pi_build_rows(const PiBuildParams p)
{
    const long long pi_s = (long long)blockIdx.x * 256 + threadIdx.x;
    if (pi_s >= p.n_local) return;
    const int pi_a = blockIdx.y;
    unsigned pi_w[PI_W];
    pi_row(p, pi_s, pi_a, pi_w);

    unsigned char* pi_t = p.table + (pi_size)pi_a * ((pi_size)PI_W * 4u * (pi_size)p.n_pad);
    #pragma unroll
    for (int k = 0; k < PI_N4; ++k)
        pi_st16(pi_t + (pi_size)k * 16u * (pi_size)p.n_pad + (pi_size)pi_s * 16u,
                pi_w[4 * k], pi_w[4 * k + 1], pi_w[4 * k + 2], pi_w[4 * k + 3]);
#if (PI_W % 4) >= 2
    pi_st8(pi_t + (pi_size)PI_N4 * 16u * (pi_size)p.n_pad + (pi_size)pi_s * 8u,
           pi_w[4 * PI_N4], pi_w[4 * PI_N4 + 1]);
#endif
#if (PI_W % 2) == 1
    pi_st4(pi_t + ((pi_size)PI_N4 * 16u + (pi_size)PI_N2 * 8u) * (pi_size)p.n_pad + (pi_size)pi_s * 4u,
           pi_w[PI_W - 1]);
#endif
}

// ---- recompute mode: the kernels that replace every read of the all-action table (DESIGN.md §8 N7) ----

// Improvement, phase 1: one thread per (local state, action = blockIdx.y).  Q = fmaf(gamma, sum_c w_c V_c, reward) with
// improve_kernel's arithmetic (expected_value, row_value_src.cuh); the state's winner is the maximum of the 64-bit key
// (Q in an order-preserving unsigned form, inverted action index), reduced with atomicMax, which does not depend on the
// order in which the actions arrive.  improve_kernel's rule, strict '>' from -1e30f in ascending action order, is
// reproduced exactly: NaN and Q <= -1e30 never compete, -0.0 is made +0.0 (the two compare equal under '>'), and among
// equal Q the lowest action has the largest inverted index.  keys[s] == 0 (nothing competed) means action 0.
// Absorbing states are skipped: they keep their action.
extern "C" __global__ void __launch_bounds__(256) pi_improve_recompute(const PiBuildParams p, const float* V, const float gamma,
                                                                       unsigned long long* keys)
{
    const long long pi_s = (long long)blockIdx.x * 256 + threadIdx.x;
    if (pi_s >= p.n_local) return;
    if (p.absorbing != nullptr && p.absorbing[pi_s]) return;
    const int pi_a = blockIdx.y;
    unsigned w[PI_W];
    pi_row(p, pi_s, pi_a, w);
    const int base = (int)w[0];
    float ev = 0.0f;
    if (base >= 0) {
        float frac[PI_D];
        int stride[PI_D];
        #pragma unroll
        for (int d = 0; d < PI_D; ++d) { frac[d] = __uint_as_float(w[1 + d]); stride[d] = p.stride[d]; }
        ev = expected_value<PI_D>(V, base, frac, stride);
    }
    float q = fmaf(gamma, ev, __uint_as_float(w[PI_D + 1]));
    if (!(q > -1.0e30f)) return;
    if (q == 0.0f) q = 0.0f;
    const unsigned u = __float_as_uint(q);
    const unsigned ord = (u & 0x80000000u) ? ~u : (u | 0x80000000u);
    atomicMax(keys + pi_s, ((unsigned long long)ord << 32) | (unsigned long long)(0xffffffffu - (unsigned)pi_a));
}

// rows[s] = row(s, policy[s]) for the local states [s_first, s_end), s_first a multiple of 32 (the regularity counters
// look at aligned groups): what compact_rows_kernel copies out of the table, at build, retrain and policy upload.  With
// `keys` it is also improvement phase 2: every state that is not absorbing takes the winner of its key first, and the
// per-block count of changed actions goes to partial[blockIdx.x], as improve_kernel writes it.
extern "C" __global__ void __launch_bounds__(256) pi_policy_rows(const PiBuildParams p, unsigned char* rows, int* policy,
                                                                 const long long s_first, const long long s_end,
                                                                 const unsigned long long* keys, unsigned* partial,
                                                                 unsigned long long* regular)
{
    const long long s = s_first + (long long)blockIdx.x * 256 + threadIdx.x;
    int changed = 0;
    int base = -2;
    if (s < s_end) {
        int a = policy[s];
        if (keys != nullptr && !(p.absorbing != nullptr && p.absorbing[s])) {
            const unsigned long long k = keys[s];
            const int best = k ? (int)(0xffffffffu - (unsigned)k) : 0;
            changed = best != a;
            a = best;
            policy[s] = best;
        }
        unsigned w[PI_W];
        pi_row(p, s, a, w);
        pi_store_row(rows, p.n_pad, s, w);
        base = (int)w[0];
    }
    count_regular_groups(base, s < s_end, regular);
    if (partial != nullptr) {
        const unsigned m = __ballot_sync(0xffffffffu, changed);
        __shared__ int s_cnt;
        if (threadIdx.x == 0) s_cnt = 0;
        __syncthreads();
        if ((threadIdx.x & 31) == 0 && m) atomicAdd(&s_cnt, __popc(m));
        __syncthreads();
        if (threadIdx.x == 0) partial[blockIdx.x] = (unsigned)s_cnt;
    }
}
)PISRC";

}  // namespace pi
