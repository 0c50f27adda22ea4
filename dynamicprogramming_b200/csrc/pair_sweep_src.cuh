// pair_sweep_src.cuh — CUDA source of the JIT generic evaluation sweeps: the gather sweep
// (policy_eval_kernel_4d/_6d of the reference, src/cuda_policy_iteration.py:616-649, :1044-1079,
// + the max|x-y| reduction :563-571, :987-995) compiled at run time by NVRTC for sm_100a with the
// grid strides baked in as immediates.  Two forms, one entry point (gp_sweep):
//
//   GP_SINGLE = 1  ONE state per thread, scalar math, the 2^D gathers issued in explicit groups of
//                  GP_G loads with the next group in flight while the fma chain consumes the current
//                  one — the default generic sweep of large 6-D grids (K5: 1.47 vs 1.68 ms per sweep
//                  for the ahead-of-time kernel; L1 data pipe 81 % busy; DESIGN.md §5)
//   GP_SINGLE = 0  TWO states per thread whose weight trees and fma chains run as one packed
//                  mul.rn.f32x2 / fma.rn.f32x2 stream (opt-in; the FMA pipe is not the limit)
//
// build.py turns this file into the string pi::kPairSweepSrc; the host prepends
//
//   GP_D        grid dimensions (>= 3)
//   GP_THREADS  threads per CTA (multiple of 32)      GP_MINB   CTAs per SM
//   GP_LV       trailing dimensions whose factors are applied per corner instead of being stored in the
//               weight tree (1..3): the tree holds 2^(D-LV) packed nodes, every corner pays LV multiplies.
//               Fewer tree registers leave more registers for gathers in flight (the sweep is latency-bound).
//   GP_G        gathers per explicitly scheduled group (0: leave the schedule to ptxas)
//   gp_off[]    V offset of corner c: sum of the storage strides of the set bits (bit d <-> dim d)
//
// and then sweep_common_src.cuh (pi::GpParams, pi::Ctl, pi::load_row, the shared device helpers).
//
// Why the packed form (DESIGN.md §5).  The scalar sweep (pi::eval_sweep_kernel) spends 2^D scalar FMUL for the
// leaf weights, 2^D-4 for the tree, 2^D FFMA for the chain and ~2^D IMAD for the gather
// addresses per state — all on the FMA pipe, where a 3-register FFMA/FMUL/IMAD issues at half
// rate on sm_100.  Here the two states of a thread share every FMA-pipe instruction (each
// half of an f32x2 op rounds exactly like the scalar op, in the reference's order
// w_c = ((((f_0 f_1) f_2) ..) f_{D-1}), ev = fma(w_c, V_c, ev), c ascending :602-613, :643-646,
// :1030-1041, :1074-1076 => bit-identical V) and the gather addresses are base + immediate.
// The gathers themselves stay scalar and fully general: nothing is assumed about the policy
// or about which dimension is stored fastest.  Lane l of warp w owns states 64 w' + l and
// 64 w' + 32 + l, so every gather instruction is still issued by 32 consecutive states
// (same coalescing as the scalar sweep), rows are read from the engine's plain storage order.

typedef unsigned long long gp_u64;

#define GP_W (GP_D + 2)
#define GP_C (1 << GP_D)
#define GP_H (GP_C / 2)
#ifndef GP_LV
#define GP_LV 1
#endif
#define GP_NT (GP_C >> GP_LV)
#ifndef GP_G
#define GP_G 0        // gathers per explicitly scheduled group (0: leave the schedule to ptxas)
#endif

__device__ __forceinline__ float gp_mul_nocse(float a, float b) {
    float r;
    asm volatile("mul.rn.f32 %0, %1, %2;" : "=f"(r) : "f"(a), "f"(b));
    return r;
}
__device__ __forceinline__ float gp_ld_ordered(const float* p) {
    float r;
    asm volatile("ld.global.nc.f32 %0, [%1];" : "=f"(r) : "l"(p));
    return r;
}

#ifndef GP_SINGLE
#define GP_SINGLE 0   // 1: one state per thread (scalar math), same immediates and explicit gather schedule
#endif

#ifndef GP_PAIRV
#define GP_PAIRV 0    // 1 (GP_SINGLE only, fast-stored dimension = logical dimension 0): gather from a PAIR SHADOW of V
#endif

#if GP_PAIRV
// P[i] = (V[i], V[i+1]): the two corners of a cell along the fast dimension are one aligned 64-bit load instead of
// two 32-bit loads that touch the same lines — half the gather requests.  Modelled on the converged K5 policy:
// 5.0 instead of 7.9 L1 wavefronts per window per warp (DESIGN.md §5).  The sweep reads pairs, and writes the plain
// value (everything else in the engine reads plain V) plus the two pair halves that contain it.
__device__ __forceinline__ float2 gp_ld_pair_ordered(const float2* p) {
    float2 r;
    asm volatile("ld.global.nc.v2.f32 {%0,%1}, [%2];" : "=f"(r.x), "=f"(r.y) : "l"(p));
    return r;
}
#endif

#if GP_SINGLE
// One state per thread: the scalar sweep (pi::eval_sweep_kernel + expected_value_grouped) with the grid's
// strides as immediates — no address arithmetic, fewer registers, more resident warps.
extern "C" __global__ void __launch_bounds__(GP_THREADS, GP_MINB) gp_sweep(const pi::GpParams p)
{
    const pi::Ctl* __restrict__ ctl = p.ctl;
    if (ctl->done) return;
    const int par = (ctl->base + p.j + ctl->parity0) & 1;
    const float* __restrict__ Vin = par ? p.V1 : p.V0;
    float* __restrict__ Vout = par ? p.V0 : p.V1;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const unsigned sched = blockIdx.x + (unsigned)p.sched_begin;
    const unsigned blk = sched + (unsigned)p.rot < (unsigned)p.n_blocks ? sched + (unsigned)p.rot : sched + (unsigned)p.rot - (unsigned)p.n_blocks;
    const long long s = (long long)blk * GP_THREADS + threadIdx.x;
    // peers need values only from the first blocks of the (rotated) schedule
    const bool peer_blk = sched < (unsigned)p.n_peer_blocks;
#if GP_PAIRV
    const float2* __restrict__ Pin = par ? p.P1 : p.P0;
    float2* __restrict__ Pout = par ? p.P0 : p.P1;
#endif
    float res = 0.0f;
    if (s < p.n_local) {
        unsigned w[GP_W];
        pi::load_row<GP_D>(p.rows, p.n_pad, s, w);
        const int b = (int)w[0];
        const float vold = Vin[p.s_begin + s];
        float vnew;
        if (b == -2) {
            vnew = vold;
        } else {
            float ev = 0.0f;
            if (b >= 0) {
                const float* v = Vin + b;
                float pre[GP_NT];
                pre[0] = 1.0f - __uint_as_float(w[1]);
                pre[1] = __uint_as_float(w[1]);
#pragma unroll
                for (int d = 1; d < GP_D - GP_LV; ++d) {
                    const float f = __uint_as_float(w[1 + d]), g = 1.0f - f;
#pragma unroll
                    for (int c = GP_NT / 2 - 1; c >= 0; --c) {
                        if (c < (1 << d)) {
                            const float t = pre[c];
                            pre[c + (1 << d)] = t * f;
                            pre[c] = t * g;
                        }
                    }
                }
                float wt[GP_LV][2];
#pragma unroll
                for (int k = 0; k < GP_LV; ++k) {
                    const float l = __uint_as_float(w[1 + GP_D - GP_LV + k]);
                    wt[k][0] = 1.0f - l;
                    wt[k][1] = l;
                }
#if GP_G == 0
#pragma unroll
                for (int c = 0; c < GP_C; ++c) {
                    float leaf = pre[c & (GP_NT - 1)];
#pragma unroll
                    for (int k = 0; k < GP_LV; ++k) leaf = leaf * wt[k][(c >> (GP_D - GP_LV + k)) & 1];
                    ev = fmaf(leaf, __ldg(v + gp_off[c]), ev);
                }
#else
                float buf[2][GP_G];
#if GP_PAIRV
                // corners 2o and 2o+1 differ in bit 0 <-> the fast dimension (stride 1): one pair load serves both
                const float2* pv = Pin + b;
#pragma unroll
                for (int i = 0; i < GP_G; i += 2) {
                    const float2 t = gp_ld_pair_ordered(pv + gp_off[i]);
                    buf[0][i] = t.x; buf[0][i + 1] = t.y;
                }
#else
#pragma unroll
                for (int i = 0; i < GP_G; ++i) buf[0][i] = gp_ld_ordered(v + gp_off[i]);
#endif
#pragma unroll
                for (int g = 0; g < GP_C / GP_G; ++g) {
                    if (g + 1 < GP_C / GP_G) {
#if GP_PAIRV
#pragma unroll
                        for (int i = 0; i < GP_G; i += 2) {
                            const float2 t = gp_ld_pair_ordered(pv + gp_off[(g + 1) * GP_G + i]);
                            buf[(g + 1) & 1][i] = t.x; buf[(g + 1) & 1][i + 1] = t.y;
                        }
#else
#pragma unroll
                        for (int i = 0; i < GP_G; ++i) buf[(g + 1) & 1][i] = gp_ld_ordered(v + gp_off[(g + 1) * GP_G + i]);
#endif
                    }
#pragma unroll
                    for (int i = 0; i < GP_G; ++i) {
                        const int c = g * GP_G + i;
                        float leaf = pre[c & (GP_NT - 1)];
#pragma unroll
                        for (int k = 0; k < GP_LV; ++k) {
                            const float f = wt[k][(c >> (GP_D - GP_LV + k)) & 1];
                            leaf = (k + 1 < GP_LV) ? gp_mul_nocse(leaf, f) : leaf * f;
                        }
                        ev = fmaf(leaf, buf[g & 1][i], ev);
                    }
                }
#endif
            }
            vnew = fmaf(p.gamma, ev, __uint_as_float(w[GP_D + 1]));
        }
        Vout[p.s_begin + s] = vnew;
#if GP_PAIRV
        {   // the two pairs that contain this value: (V[g], V[g+1]).x and (V[g-1], V[g]).y
            const long long g = p.s_begin + s;
            Pout[g].x = vnew;
            if (g > 0) Pout[g - 1].y = vnew;
        }
#endif
        if (peer_blk) pi::store_peers(p.peers, par != 0, p.s_begin + s, vnew);
        res = fabsf(vnew - vold);
    }
    if (!p.check) return;
    __shared__ float s_red[32];
    res = pi::warp_max(res);
    if (lane == 0) s_red[warp] = res;
    __syncthreads();
    if (threadIdx.x < 32) {
        float r = threadIdx.x < GP_THREADS / 32 ? s_red[threadIdx.x] : 0.0f;
        r = pi::warp_max(r);
        if (threadIdx.x == 0) p.partial[sched] = r;
    }
}
#else
extern "C" __global__ void __launch_bounds__(GP_THREADS, GP_MINB) gp_sweep(const pi::GpParams p)
{
    const pi::Ctl* __restrict__ ctl = p.ctl;
    if (ctl->done) return;
    const int par = (ctl->base + p.j + ctl->parity0) & 1;
    const float* __restrict__ Vin = par ? p.V1 : p.V0;
    float* __restrict__ Vout = par ? p.V0 : p.V1;

    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const long long sA = ((long long)blockIdx.x * (GP_THREADS / 32) + warp) * 64 + lane;
    const long long sB = sA + 32;
    const bool inA = sA < p.n_local, inB = sB < p.n_local;
    float res = 0.0f;

    if (inA) {
        unsigned wA[GP_W], wB[GP_W];
        pi::load_row<GP_D>(p.rows, p.n_pad, sA, wA);
        if (inB) pi::load_row<GP_D>(p.rows, p.n_pad, sB, wB);
        else {
#pragma unroll
            for (int k = 0; k < GP_W; ++k) wB[k] = k == 0 ? 0xfffffffeu : 0u;
        }
        const float voldA = Vin[p.s_begin + sA];
        const float voldB = inB ? Vin[p.s_begin + sB] : 0.0f;
        const int bA = (int)wA[0], bB = (int)wB[0];
        // sentinel rows gather from a valid address and are discarded afterwards
        const float* vA = Vin + (bA >= 0 ? bA : 0);
        const float* vB = Vin + (bB >= 0 ? bB : 0);

        // weight tree over dims 0..D-1-LV, packed (state A, state B)
        gp_u64 node[GP_NT];
        {
            const float fa = __uint_as_float(wA[1]), fb = __uint_as_float(wB[1]);
            node[0] = pi::pk(1.0f - fa, 1.0f - fb);
            node[1] = pi::pk(fa, fb);
#pragma unroll
            for (int d = 1; d < GP_D - GP_LV; ++d) {
                const float xa = __uint_as_float(wA[1 + d]), xb = __uint_as_float(wB[1 + d]);
                const gp_u64 f = pi::pk(xa, xb), g = pi::pk(1.0f - xa, 1.0f - xb);
#pragma unroll
                for (int c = GP_NT / 2 - 1; c >= 0; --c) {   // constant trip count: node[] stays in registers
                    if (c < (1 << d)) {
                        const gp_u64 t = node[c];
                        node[c + (1 << d)] = pi::mul2(t, f);
                        node[c] = pi::mul2(t, g);
                    }
                }
            }
        }
        // factors of the trailing dimensions D-LV .. D-1: wt[k][bit]
        gp_u64 wt[GP_LV][2];
#pragma unroll
        for (int k = 0; k < GP_LV; ++k) {
            const float la = __uint_as_float(wA[1 + GP_D - GP_LV + k]), lb = __uint_as_float(wB[1 + GP_D - GP_LV + k]);
            wt[k][0] = pi::pk(1.0f - la, 1.0f - lb);
            wt[k][1] = pi::pk(la, lb);
        }

        gp_u64 ev = pi::pk(0.0f, 0.0f);
#if GP_G == 0
#pragma unroll
        for (int c = 0; c < GP_C; ++c) {
            gp_u64 leaf = node[c & (GP_NT - 1)];
#pragma unroll
            for (int k = 0; k < GP_LV; ++k) {
                const gp_u64 f = wt[k][(c >> (GP_D - GP_LV + k)) & 1];
                leaf = (k + 1 < GP_LV) ? pi::mul2_nocse(leaf, f) : pi::mul2(leaf, f);
            }
            ev = pi::fma2(leaf, pi::pk(__ldg(vA + gp_off[c]), __ldg(vB + gp_off[c])), ev);
        }
#else
        // explicitly scheduled gathers (see pi::expected_value_grouped): groups of GP_G corners, the loads of
        // group g+1 are issued (volatile: in order) before the fma chain of group g consumes its values
        float bufA[2][GP_G], bufB[2][GP_G];
#pragma unroll
        for (int i = 0; i < GP_G; ++i) { bufA[0][i] = gp_ld_ordered(vA + gp_off[i]); bufB[0][i] = gp_ld_ordered(vB + gp_off[i]); }
#pragma unroll
        for (int g = 0; g < GP_C / GP_G; ++g) {
            if (g + 1 < GP_C / GP_G) {
#pragma unroll
                for (int i = 0; i < GP_G; ++i) {
                    bufA[(g + 1) & 1][i] = gp_ld_ordered(vA + gp_off[(g + 1) * GP_G + i]);
                    bufB[(g + 1) & 1][i] = gp_ld_ordered(vB + gp_off[(g + 1) * GP_G + i]);
                }
            }
#pragma unroll
            for (int i = 0; i < GP_G; ++i) {
                const int c = g * GP_G + i;
                gp_u64 leaf = node[c & (GP_NT - 1)];
#pragma unroll
                for (int k = 0; k < GP_LV; ++k) {
                    const gp_u64 f = wt[k][(c >> (GP_D - GP_LV + k)) & 1];
                    leaf = (k + 1 < GP_LV) ? pi::mul2_nocse(leaf, f) : pi::mul2(leaf, f);
                }
                ev = pi::fma2(leaf, pi::pk(bufA[g & 1][i], bufB[g & 1][i]), ev);
            }
        }
#endif
        float evA, evB;
        pi::unpk(ev, evA, evB);
        // sentinel rows: terminated (-1) -> sum := 0 (:231-232); absorbing (-2) -> new_V := V (:221)
        const float vnewA = bA == -2 ? voldA : fmaf(p.gamma, bA >= 0 ? evA : 0.0f, __uint_as_float(wA[GP_D + 1]));
        Vout[p.s_begin + sA] = vnewA;
        if (p.peers.n) pi::store_peers(p.peers, par != 0, p.s_begin + sA, vnewA);
        res = fabsf(vnewA - voldA);
        if (inB) {
            const float vnewB = bB == -2 ? voldB : fmaf(p.gamma, bB >= 0 ? evB : 0.0f, __uint_as_float(wB[GP_D + 1]));
            Vout[p.s_begin + sB] = vnewB;
            if (p.peers.n) pi::store_peers(p.peers, par != 0, p.s_begin + sB, vnewB);
            res = fmaxf(res, fabsf(vnewB - voldB));
        }
    }
    if (!p.check) return;
    __shared__ float s_red[32];
    res = pi::warp_max(res);
    if (lane == 0) s_red[warp] = res;
    __syncthreads();
    if (threadIdx.x < 32) {
        float r = threadIdx.x < GP_THREADS / 32 ? s_red[threadIdx.x] : 0.0f;
        r = pi::warp_max(r);
        if (threadIdx.x == 0) p.partial[blockIdx.x] = r;
    }
}
#endif   // GP_SINGLE
