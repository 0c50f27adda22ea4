// xline_sweep_src.cuh — CUDA source of the x-line evaluation sweep (policy_eval_kernel_4d/_6d
// of the reference, src/cuda_policy_iteration.py:616-649, :1044-1079, + the max|x-y|
// reduction :563-571, :987-995), compiled at run time by NVRTC for sm_100a with the grid
// geometry baked in as constants.  build.py turns this file into the string
// pi::kXlineSweepSrc (xline_sweep_src.inc); the host prepends a preamble that defines
//
//   XL_D        grid dimensions (>= 3; the fast-stored dimension is logical dimension 0)
//   XL_K        consecutive states along the fast dimension per thread (2 or 4)
//   XL_S        length of an x-line (shape of the fast dimension), XL_S % XL_K == 0
//   XL_LV       0: weight tree over dims 0..D-2 held in registers; 1: dims 0..D-3
//   XL_PF       window loads kept in flight per thread
//   XL_ROLL     run-time iterations the 2^(D-1) windows are split into (1, 2; 4 with XL_LV == 1)
//   XL_NL       x-lines per tile        XL_WARPS   warps per CTA       XL_MINB  CTAs per SM
//   xl_woff[]   V offset of window o (sum of the strides of the set dimensions, bit d-1 <-> dim d)
//   xl_stride[] V stride of logical dimension d
//   xl_ntile[], xl_tline[]   tiles per storage position / V-line step between tiles
//   xl_line_off[]            V-line offset of x-line xl inside a tile (__constant__)
//
// and then sweep_common_src.cuh (pi::XlParams, pi::Ctl, the shared device helpers).
//
// Design (DESIGN.md §5).  A thread owns K consecutive states of one x-line.  When their
// successor cells are consecutive (base_j = A + j — the translation-invariant case the
// layout probe picks the fast dimension for) the 2^D corners of all K states live in
// 2^(D-1) windows V[A + woff_o .. A + woff_o + K]: ONE aligned 128/64-bit load per window
// plus one shuffle for the element shared with the neighbouring lane, instead of K * 2
// scalar gathers.  Weights and fma chains of two states are evaluated as packed
// mul.rn.f32x2 / fma.rn.f32x2 (FMUL2 / FFMA2) — every half rounds exactly like the scalar
// instruction, in the reference's order w_c = ((((f_0 f_1) f_2) ..) f_{D-1}),
// ev = fma(w_c, V_c, ev), c ascending (:602-613, :643-646, :1030-1041, :1074-1076), so V
// is bit-identical.  Anything irregular (clamped / wrapped successors, mixed sentinels)
// takes the scalar path with the same arithmetic.
//
// Rows are word-SoA in tile order (one persistent CTA walks tiles blockIdx, +gridDim, ..):
// the gathers of a tile stay inside a compact box of V (L1 reuse) while the row stream is
// one coalesced 128-bit load per word, prefetched into L2 one tile ahead by TMA.

typedef unsigned long long xl_u64;

#define XL_W (XL_D + 2)
#define XL_TPL (XL_S / XL_K)          // threads per x-line
#define XL_LPW (32 / XL_TPL)          // x-lines per warp
#define XL_NO (1 << (XL_D - 1))       // windows per state group
#define XL_NH (XL_NO / 2)
#define XL_DT (XL_D - 1 - XL_LV)      // dims held in the stored weight tree
#define XL_NN (1 << XL_DT)
#define XL_NP (XL_K / 2)

struct XlVec {
    float v[XL_K];
    __device__ __forceinline__ void load(const float* p) {
#if XL_K == 4
        const float4 t = __ldg(reinterpret_cast<const float4*>(p));
        v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
#else
        const float2 t = __ldg(reinterpret_cast<const float2*>(p));
        v[0] = t.x; v[1] = t.y;
#endif
    }
};

// Scalar expected value of one state (reference order; one copy of the code).
__device__ __noinline__ float xl_expected_value_scalar(const float* __restrict__ V, int base, const float* fr) {
    float pre[XL_NO];
    pre[0] = 1.0f - fr[0];
    pre[1] = fr[0];
#pragma unroll
    for (int d = 1; d < XL_D - 1; ++d) {
        const float f = fr[d], g = 1.0f - f;
#pragma unroll
        for (int c = XL_NO / 2 - 1; c >= 0; --c) {
            if (c < (1 << d)) {
                const float t = pre[c];
                pre[c + (1 << d)] = t * f;
                pre[c] = t * g;
            }
        }
    }
    const float fl = fr[XL_D - 1], gl = 1.0f - fl;
    const float* v = V + base;
    float ev = 0.0f;
#pragma unroll
    for (int c = 0; c < 2 * XL_NO; ++c) {
        const int xb = c & 1, o = c >> 1;                 // bit 0 <-> dimension 0 (stride 1)
        const float w = pre[c & (XL_NO - 1)] * ((c >> (XL_D - 1)) ? fl : gl);
        ev = fmaf(w, __ldg(v + xl_woff[o] + xb), ev);
    }
    return ev;
}

// Window path of one thread (all lanes of the warp execute it: shuffles).
//   DELTA = 1: the thread's vector starts at A, the extra element is the first of the next lane's vector
//   DELTA = 0: the vector starts at A + 1, the extra element is the last of the previous lane's vector
template <int DELTA>
__device__ __forceinline__ void xl_window_path(const float* __restrict__ vb, const float (&frac)[XL_K][XL_D],
                                               float (&ev_out)[XL_K]) {
    xl_u64 node[XL_NP][XL_NN];
    xl_u64 wl[XL_NP][2], wm[XL_NP][2];
#pragma unroll
    for (int q = 0; q < XL_NP; ++q) {
        const float fa = frac[2 * q][0], fb = frac[2 * q + 1][0];
        node[q][0] = pi::pk(1.0f - fa, 1.0f - fb);
        node[q][1] = pi::pk(fa, fb);
#pragma unroll
        for (int d = 1; d < XL_DT; ++d) {
            const xl_u64 f = pi::pk(frac[2 * q][d], frac[2 * q + 1][d]);
            const xl_u64 g = pi::pk(1.0f - frac[2 * q][d], 1.0f - frac[2 * q + 1][d]);
#pragma unroll
            for (int c = XL_NN / 2 - 1; c >= 0; --c) {   // constant trip count: node[] stays in registers
                if (c < (1 << d)) {
                    const xl_u64 t = node[q][c];
                    node[q][c + (1 << d)] = pi::mul2(t, f);
                    node[q][c] = pi::mul2(t, g);
                }
            }
        }
        wl[q][0] = pi::pk(1.0f - frac[2 * q][XL_D - 1], 1.0f - frac[2 * q + 1][XL_D - 1]);
        wl[q][1] = pi::pk(frac[2 * q][XL_D - 1], frac[2 * q + 1][XL_D - 1]);
        wm[q][0] = pi::pk(1.0f - frac[2 * q][XL_D - 2], 1.0f - frac[2 * q + 1][XL_D - 2]);
        wm[q][1] = pi::pk(frac[2 * q][XL_D - 2], frac[2 * q + 1][XL_D - 2]);
    }

    xl_u64 ev[XL_NP];
#pragma unroll
    for (int q = 0; q < XL_NP; ++q) ev[q] = pi::pk(0.0f, 0.0f);

    // The 2^(D-1) windows are walked as XL_ROLL run-time iterations of XL_NB fully unrolled
    // windows (the rolled loop bounds code size and the live ranges of the in-flight loads;
    // the stored tree is indexed by compile-time constants only).  A ring of XL_PF vector
    // loads stays in flight across iteration boundaries.
    constexpr int NB = XL_NO / XL_ROLL;
    static_assert(XL_PF <= NB, "XL_PF must not exceed the windows per rolled iteration");
    static_assert(XL_LV == 0 ? (XL_ROLL == 1 || XL_ROLL == 2) : (XL_ROLL == 1 || XL_ROLL == 2 || XL_ROLL == 4),
                  "unsupported XL_ROLL for this XL_LV");
    XlVec ring[XL_PF];
#pragma unroll
    for (int i = 0; i < XL_PF; ++i) ring[i].load(vb + xl_woff[i]);
#pragma unroll 1
    for (int r = 0; r < XL_ROLL; ++r) {
        const float* vr = vb + xl_woff[r * NB];
        const float* vn = vb + xl_woff[(r + 1 < XL_ROLL ? r + 1 : r) * NB];   // next iteration's windows
        const bool more = r + 1 < XL_ROLL;
        // last-dimension / level D-2 factors of this iteration
        xl_u64 wls[XL_NP], wms[XL_NP];
#pragma unroll
        for (int q = 0; q < XL_NP; ++q) {
            if (XL_ROLL == 1) { wls[q] = wl[q][0]; wms[q] = wm[q][0]; }
            else {
                const int half = (r * NB) / XL_NH;
                wls[q] = half ? wl[q][1] : wl[q][0];
                const int mb = ((r * NB) % XL_NH) / (XL_NH / 2);
                wms[q] = mb ? wm[q][1] : wm[q][0];
            }
        }
#pragma unroll
        for (int ob = 0; ob < NB; ++ob) {
            const XlVec own = ring[ob % XL_PF];
            if (ob + XL_PF < NB) ring[ob % XL_PF].load(vr + (xl_woff[ob + XL_PF] - xl_woff[0]));
            else if (XL_ROLL > 1) { if (more) ring[ob % XL_PF].load(vn + xl_woff[ob + XL_PF - NB]); }
            float W[XL_K + 1];
            if (DELTA) {
#pragma unroll
                for (int k = 0; k < XL_K; ++k) W[k] = own.v[k];
                W[XL_K] = __shfl_down_sync(0xffffffffu, own.v[0], 1);
            } else {
                W[0] = __shfl_up_sync(0xffffffffu, own.v[XL_K - 1], 1);
#pragma unroll
                for (int k = 0; k < XL_K; ++k) W[k + 1] = own.v[k];
            }
            // o = r * NB + ob;  half = o / NH,  ol = o % NH
#pragma unroll
            for (int xb = 0; xb < 2; ++xb) {
#pragma unroll
                for (int q = 0; q < XL_NP; ++q) {
                    xl_u64 leaf;
                    if (XL_ROLL == 1) {
                        const int half = ob / XL_NH, ol = ob % XL_NH;
#if XL_LV == 0
                        leaf = pi::mul2(node[q][2 * ol + xb], wl[q][half]);
#else
                        leaf = pi::mul2(pi::mul2_nocse(node[q][2 * (ol % (XL_NH / 2)) + xb], wm[q][ol / (XL_NH / 2)]), wl[q][half]);
#endif
                    } else {
#if XL_LV == 0
                        leaf = pi::mul2(node[q][2 * ob + xb], wls[q]);                       // NB == NH: ol == ob
#else
                        if (NB == XL_NH) leaf = pi::mul2(pi::mul2_nocse(node[q][2 * (ob % (XL_NH / 2)) + xb], wm[q][ob / (XL_NH / 2)]), wls[q]);
                        else leaf = pi::mul2(pi::mul2_nocse(node[q][2 * ob + xb], wms[q]), wls[q]);   // NB == NH/2
#endif
                    }
                    ev[q] = pi::fma2(leaf, pi::pk(W[2 * q + xb], W[2 * q + 1 + xb]), ev[q]);
                }
            }
        }
    }
#pragma unroll
    for (int q = 0; q < XL_NP; ++q) pi::unpk(ev[q], ev_out[2 * q], ev_out[2 * q + 1]);
}

extern "C" __global__ void __launch_bounds__(XL_WARPS * 32, XL_MINB) xl_sweep(const pi::XlParams p)
{
    const pi::Ctl* __restrict__ ctl = p.ctl;
    if (ctl->done) return;
    const int par = (ctl->base + p.j + ctl->parity0) & 1;
    const float* __restrict__ Vin = par ? p.V1 : p.V0;
    float* __restrict__ Vout = par ? p.V0 : p.V1;

    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int li = lane / XL_TPL;
    const int xl = warp * XL_LPW + li;
    const int x0 = (lane - li * XL_TPL) * XL_K;
    const bool active = li < XL_LPW && xl < XL_NL;
    const long long my_line_off = active ? xl_line_off[xl] : 0;
    const unsigned full = 0xffffffffu;
    float res = 0.0f;
    unsigned n_win = 0, n_sca = 0;

    for (long long tile = blockIdx.x; tile < p.n_tiles; tile += gridDim.x) {
        if (p.prefetch && threadIdx.x == 0 && tile + gridDim.x < p.n_tiles) {
            const unsigned* nx = p.rows + (size_t)(tile + gridDim.x) * (size_t)(XL_NL * XL_S);
#pragma unroll
            for (int k = 0; k < XL_W; ++k)
                asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(nx + (size_t)k * (size_t)p.plane_words),
                             "r"((unsigned)(XL_NL * XL_S * 4)) : "memory");
        }
        // tile -> V line of its origin (constant divisors)
        long long origin = 0;
        {
            unsigned t = (unsigned)(p.tile_begin + tile);
#pragma unroll
            for (int k = XL_D - 2; k >= 0; --k) {
                const unsigned q = t / (unsigned)xl_ntile[k];
                origin += (long long)(t - q * (unsigned)xl_ntile[k]) * xl_tline[k];
                t = q;
            }
        }
        unsigned w[XL_W][XL_K];
        float vold[XL_K];
        bool live[XL_K];
        long long v0 = 0, B = 0;
        bool use = false, scalar = false;
        int delta = 0;
#pragma unroll
        for (int j = 0; j < XL_K; ++j) { live[j] = false; vold[j] = 0.0f; }
#pragma unroll
        for (int k = 0; k < XL_W; ++k)
#pragma unroll
            for (int j = 0; j < XL_K; ++j) w[k][j] = k == 0 ? 0xfffffffeu : 0u;   // idle lanes: absorbing rows

        if (active) {
            const size_t r0 = ((size_t)tile * XL_NL + xl) * XL_S + x0;
#pragma unroll
            for (int k = 0; k < XL_W; ++k) {
                const unsigned* src = p.rows + (size_t)k * (size_t)p.plane_words + r0;
#if XL_K == 4
                const uint4 t = pi::ld_stream16(src);
                w[k][0] = t.x; w[k][1] = t.y; w[k][2] = t.z; w[k][3] = t.w;
#else
                const uint2 t = pi::ld_stream8(src);
                w[k][0] = t.x; w[k][1] = t.y;
#endif
            }
            v0 = (origin + my_line_off) * XL_S + x0;
            XlVec vo;
            vo.load(Vin + v0);
#pragma unroll
            for (int j = 0; j < XL_K; ++j) vold[j] = vo.v[j];

            // consecutive-successor test: every live state must have base_j - j == A
            int A = 0;
            bool have = false, ok = true;
#pragma unroll
            for (int j = 0; j < XL_K; ++j) {
                const int b = (int)w[0][j];
                live[j] = b >= 0;
                if (live[j]) {
                    if (!have) { A = b - j; have = true; }
                    else if (b - j != A) ok = false;
                }
            }
            if (have) {
                const int m = A & (XL_K - 1);   // two's complement: also right for A = -1..-K+1
                if (ok && m == 0) { delta = 1; B = A; use = true; }
                else if (ok && m == XL_K - 1) { delta = 0; B = A + 1; use = true; }
                else scalar = true;
            }
        }

        // one window orientation per warp: the minority takes the scalar path
        const unsigned m1 = __ballot_sync(full, use && delta == 1);
        const unsigned m0 = __ballot_sync(full, use && delta == 0);
        const int wdelta = __popc(m1) >= __popc(m0) ? 1 : 0;
        if (use && delta != wdelta) { use = false; scalar = true; }
        // `own` lanes stream their own windows (their vectors feed the neighbours' extra
        // elements); a lane whose extra element is NOT in its neighbour's vector still
        // streams, but takes its result from the scalar path.
        const bool own = use;
        {
            const int Bi = own ? (int)B : -1000;
            const int Bn = wdelta ? __shfl_down_sync(full, Bi, 1) : __shfl_up_sync(full, Bi, 1);
            const bool lane_ok = wdelta ? (lane < 31 && Bn == (int)B + XL_K) : (lane > 0 && Bn == (int)B - XL_K);
            const bool need_edge = use && (wdelta ? live[XL_K - 1] : live[0]);
            if (need_edge && !lane_ok) { use = false; scalar = true; }
        }
        const unsigned mo = __ballot_sync(full, own);

        float ev[XL_K];
#pragma unroll
        for (int j = 0; j < XL_K; ++j) ev[j] = 0.0f;

        if (mo) {   // warp-uniform
            float frac[XL_K][XL_D];
#pragma unroll
            for (int j = 0; j < XL_K; ++j)
#pragma unroll
                for (int d = 0; d < XL_D; ++d) frac[j][d] = __uint_as_float(w[1 + d][j]);
            // lanes without windows of their own re-load those of the first lane that has some
            const int Bw = __shfl_sync(full, (int)B, __ffs(mo) - 1);
            const float* vb = Vin + (own ? (int)B : Bw);
            float evw[XL_K];
            if (wdelta) xl_window_path<1>(vb, frac, evw);
            else xl_window_path<0>(vb, frac, evw);
            if (use) {
#pragma unroll
                for (int j = 0; j < XL_K; ++j) ev[j] = evw[j];
            }
        }
        if (scalar) {
#pragma unroll 1
            for (int j = 0; j < XL_K; ++j) {
                int b = 0;
                float fr[XL_D];
#pragma unroll
                for (int jj = 0; jj < XL_K; ++jj)
                    if (jj == j) {
                        b = (int)w[0][jj];
#pragma unroll
                        for (int d = 0; d < XL_D; ++d) fr[d] = __uint_as_float(w[1 + d][jj]);
                    }
                float e = 0.0f;
                if (b >= 0) e = xl_expected_value_scalar(Vin, b, fr);
#pragma unroll
                for (int jj = 0; jj < XL_K; ++jj)
                    if (jj == j) ev[jj] = e;
            }
        }
        n_win += use ? 1u : 0u;
        n_sca += scalar ? 1u : 0u;

        if (active) {
            float vnew[XL_K];
#pragma unroll
            for (int j = 0; j < XL_K; ++j) {
                const int b = (int)w[0][j];
                // sentinel rows: terminated (-1) -> sum := 0 (:231-232); absorbing (-2) -> new_V := V (:221)
                vnew[j] = b == -2 ? vold[j] : fmaf(p.gamma, b >= 0 ? ev[j] : 0.0f, __uint_as_float(w[XL_D + 1][j]));
                res = fmaxf(res, fabsf(vnew[j] - vold[j]));
            }
#if XL_K == 4
            *reinterpret_cast<float4*>(Vout + v0) = make_float4(vnew[0], vnew[1], vnew[2], vnew[3]);
#else
            *reinterpret_cast<float2*>(Vout + v0) = make_float2(vnew[0], vnew[1]);
#endif
            if (p.peers.n) {
#pragma unroll
                for (int j = 0; j < XL_K; ++j) pi::store_peers(p.peers, par != 0, v0 + j, vnew[j]);
            }
        }
    }

    if (p.stats) {
        const unsigned a = __reduce_add_sync(full, n_win), b = __reduce_add_sync(full, n_sca);
        if (lane == 0) { atomicAdd(p.stats, (unsigned long long)a); atomicAdd(p.stats + 1, (unsigned long long)b); }
    }
    if (!p.check) return;
    __shared__ float s_red[32];
    res = pi::warp_max(res);
    if (lane == 0) s_red[warp] = res;
    __syncthreads();
    if (threadIdx.x < 32) {
        float r = threadIdx.x < XL_WARPS ? s_red[threadIdx.x] : 0.0f;
        r = pi::warp_max(r);
        if (threadIdx.x == 0) p.partial[blockIdx.x] = r;
    }
}
