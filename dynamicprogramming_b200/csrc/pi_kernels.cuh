// pi_kernels.cuh — ahead-of-time sm_100a kernels of the policy-iteration engine.
//
// Everything here works on *compact transition rows*: for one (state, action)
// pair a row is W = D + 2 32-bit words
//     [ base | frac_0 .. frac_{D-1} | reward ]
// where `base` is the flat index of the lower corner of the interpolation cell
// (or a PI_ROW_* sentinel) and frac_d the position inside the cell.  The 2^D
// corner indices and weights of the reference's get_barycentric_{2,4,6}d
// (src/cuda_policy_iteration.py:183-210, :580-614, :1007-1042) are rebuilt in
// registers with the reference's exact operation order, so results are
// bit-identical while a 6-D row costs 32 B of HBM instead of 516 B.
//
// Row storage ("plane-SoA"): the W words of a row are split into 16-byte,
// 8-byte and 4-byte planes; plane p of a table holding n_pad states is one
// contiguous array, so lane i of a warp reads/writes 16 B at stride 16 B:
// every row access is a fully coalesced 128-bit (or 64/32-bit) transaction.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#define PI_ROW_TERMINATED (-1)
#define PI_ROW_ABSORBING (-2)

namespace pi {

constexpr int kBlock = 256;
constexpr int kMaxDims = 6;

// ---------------------------------------------------------------------------
// Device control block: lets a stream of identical sweep launches sequence
// itself (sweep counter, ping-pong parity, residual, convergence flag) with no
// host round trip per sweep.  Mirrors the loop state of policy_evaluation()
// (src/cuda_policy_iteration.py:300-336).
// ---------------------------------------------------------------------------
struct Ctl {
    int base;                   // sweeps completed before the batch in flight
    int parity0;                // V buffer that was "current" when the evaluation started
    int done;                   // 1 once a sync-point residual was < theta
    int conv_sweep;             // index i of the sweep at which the evaluation converged
    float last_delta;           // residual of the last examined sweep (local to this rank)
    float check_delta;          // residual examined at the last sync point (global)
    unsigned long long changed; // improvement: states whose action changed (local)
    unsigned int pad[8];
};

// Grid geometry.  `stride` is the reference's row-major flat index (dim 0 slowest,
// what callers see); `istride` is the engine's INTERNAL storage order, in which one
// chosen dimension (`perm[n_dims-1]`) is made the fastest so that the 32 lanes of a
// warp gather from neighbouring addresses (see DESIGN.md §3).  perm[k] = logical
// dimension stored at position k (0 = slowest).  Arithmetic never depends on it.
struct GridDesc {
    int n_dims;
    int shape[kMaxDims];
    int stride[kMaxDims];
    int istride[kMaxDims];
    int perm[kMaxDims];
    float lo[kMaxDims];
    float hi[kMaxDims];
};

__host__ __device__ inline long long internal_to_ref(const GridDesc& g, long long s_int) {
    long long r = s_int, ref = 0;
    for (int k = g.n_dims - 1; k >= 0; --k) {
        const int d = g.perm[k];
        const long long q = r / g.shape[d];
        ref += (r - q * g.shape[d]) * (long long)g.stride[d];
        r = q;
    }
    return ref;
}
__host__ __device__ inline long long ref_to_internal(const GridDesc& g, long long s_ref) {
    long long r = s_ref, out = 0;
    for (int d = g.n_dims - 1; d >= 0; --d) {
        const long long q = r / g.shape[d];
        out += (r - q * g.shape[d]) * (long long)g.istride[d];
        r = q;
    }
    return out;
}

// ---------------------------------------------------------------------------
// Sharded runs: fused V exchange.  Every evaluation-sweep kernel stores a new value not only into
// its own V buffer but also, through peer pointers (CUDA IPC over NVLink / NVSwitch), directly into
// the V buffer of every rank whose transition rows reference that state (`[lo, hi)` = the sub-range
// of THIS rank's slice that peer r needs, computed once after the table build).  The transfer
// overlaps the sweep tile by tile; a sweep ends with xgpu_barrier_kernel instead of an NCCL
// send/recv group.  Replaces nothing in the reference (single GPU); SURVEY §5 / §8(e).
// ---------------------------------------------------------------------------
constexpr int kMaxPeers = 7;
struct PeerOut {
    int n;
    int pad;
    float* V0[kMaxPeers];
    float* V1[kMaxPeers];
    long long lo[kMaxPeers];
    long long hi[kMaxPeers];
};

// out_is_V0: the sweep writes buffer 0 (of every rank) this time
// Fully unrolled over the (few) entries: a run-time-indexed loop over a kernel-parameter struct makes the compiler copy
// the struct to local memory and turns every range test into local loads (measured at N = 2: +34 us per K5 sweep in the
// gather sweep, +71 us in the plane-staged sweep, before any byte crossed NVLink).
__device__ __forceinline__ void store_peers(const PeerOut& po, bool out_is_V0, long long g, float v) {
#pragma unroll
    for (int r = 0; r < kMaxPeers; ++r)
        if (r < po.n && g >= po.lo[r] && g < po.hi[r]) (out_is_V0 ? po.V0[r] : po.V1[r])[g] = v;
}

// Cross-GPU barrier at the end of a sweep: thread t publishes this rank's epoch into rank t's flag
// array (release, system scope — the sweep kernel before it in stream order has completed, so its
// peer stores are performed), then waits until rank t's epoch has arrived in the local array.
// Only ranks that exchange values take part (`partners`): with contiguous ranges of the slowest-stored
// dimension that is the two neighbours (plus the wrap-around partner of a periodic angle), not all 7
// peers, so a sweep waits for the slowest of 3 ranks instead of the slowest of 8.
// flags_local[r] is written only by rank r.  A rank that never arrives (crashed peer) trips the
// timeout instead of hanging the GPU; the host turns err != 0 into PI_ERR_COMM.
struct BarrierParams {
    unsigned* flags_local;
    unsigned* flags_peer[kMaxPeers + 1];   // indexed by rank; [own rank] unused
    unsigned* epoch;                       // local sweep counter
    unsigned* err;
    Ctl* ctl;                              // a timeout also sets ctl->done: the remaining sweeps of the batch become no-ops
    long long timeout_ticks;               // clock64 ticks a rank waits for a peer (DPB200_BARRIER_TIMEOUT_S, default 120 s)
    int rank;
    int world;
    unsigned partners;                     // bit r: rank r exchanges values with this rank (either direction); only those
                                           // pairs synchronise — the relation is symmetric, both sides compute it from the plan
};
__global__ void xgpu_barrier_kernel(const BarrierParams b) {
    const int t = threadIdx.x;
    const unsigned e = *b.epoch + 1;
    if (*b.err) return;   // a barrier already timed out in this call: do not wait again, the host reports PI_ERR_COMM
    if (t < b.world && t != b.rank && ((b.partners >> t) & 1u)) {
        __threadfence_system();
        asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(b.flags_peer[t] + b.rank), "r"(e) : "memory");
        const long long t0 = clock64();
        unsigned seen;
        do {
            asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(seen) : "l"(b.flags_local + t) : "memory");
            if ((int)(seen - e) >= 0) break;
            if (clock64() - t0 > b.timeout_ticks) {   // never compute on stale halo values
                *b.err = 1u;
                b.ctl->done = 1;
                break;
            }
        } while (true);
    }
    __syncthreads();
    if (t == 0) *b.epoch = e;
}

// ---------------------------------------------------------------------------
// Row layout helpers
// ---------------------------------------------------------------------------
template <int D>
struct Row {
    static constexpr int W = D + 2;
    static constexpr int N4 = W / 4;        // 16-byte planes
    static constexpr int N2 = (W % 4) / 2;  // 8-byte plane (0/1)
    static constexpr int N1 = W % 2;        // 4-byte plane (0/1)
    static constexpr int kBytes = W * 4;
};

__host__ __device__ inline size_t row_table_bytes(int D, long long n_pad) {
    return (size_t)(D + 2) * 4u * (size_t)n_pad;
}

// streaming (read-once) loads: do not pollute L1, mark evict-first in L2
__device__ __forceinline__ uint4 ld_stream16(const void* p) {
    uint4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
                 : "l"(p));
    return r;
}
__device__ __forceinline__ uint2 ld_stream8(const void* p) {
    uint2 r;
    asm volatile("ld.global.nc.L1::no_allocate.v2.u32 {%0,%1}, [%2];"
                 : "=r"(r.x), "=r"(r.y)
                 : "l"(p));
    return r;
}
__device__ __forceinline__ unsigned ld_stream4(const void* p) {
    unsigned r;
    asm volatile("ld.global.nc.L1::no_allocate.u32 %0, [%1];" : "=r"(r) : "l"(p));
    return r;
}
__device__ __forceinline__ void st_stream16(void* p, uint4 v) {
    asm volatile("st.global.L1::no_allocate.v4.u32 [%0], {%1,%2,%3,%4};" ::"l"(p), "r"(v.x), "r"(v.y),
                 "r"(v.z), "r"(v.w)
                 : "memory");
}
__device__ __forceinline__ void st_stream8(void* p, uint2 v) {
    asm volatile("st.global.L1::no_allocate.v2.u32 [%0], {%1,%2};" ::"l"(p), "r"(v.x), "r"(v.y) : "memory");
}
__device__ __forceinline__ void st_stream4(void* p, unsigned v) {
    asm volatile("st.global.L1::no_allocate.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}

// L2 eviction policies (createpolicy): the row stream is read once per sweep and should leave the L2
// first; the gathered V window is re-read by neighbouring blocks and should stay.
__device__ __forceinline__ unsigned long long l2_policy_evict_first() {
    unsigned long long pol;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
    return pol;
}
__device__ __forceinline__ unsigned long long l2_policy_evict_last() {
    unsigned long long pol;
    asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(pol));
    return pol;
}
__device__ __forceinline__ uint4 ld_stream16_hint(const void* p, unsigned long long pol) {
    uint4 r;
    asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.v4.u32 {%0,%1,%2,%3}, [%4], %5;"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
                 : "l"(p), "l"(pol));
    return r;
}
__device__ __forceinline__ uint2 ld_stream8_hint(const void* p, unsigned long long pol) {
    uint2 r;
    asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.v2.u32 {%0,%1}, [%2], %3;"
                 : "=r"(r.x), "=r"(r.y)
                 : "l"(p), "l"(pol));
    return r;
}
__device__ __forceinline__ unsigned ld_stream4_hint(const void* p, unsigned long long pol) {
    unsigned r;
    asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.u32 %0, [%1], %2;" : "=r"(r) : "l"(p), "l"(pol));
    return r;
}
__device__ __forceinline__ float ld_keep4(const float* p, unsigned long long pol) {
    float r;
    asm volatile("ld.global.nc.L2::cache_hint.f32 %0, [%1], %2;" : "=f"(r) : "l"(p), "l"(pol));
    return r;
}

// load_row with an L2 eviction policy on every plane
template <int D>
__device__ __forceinline__ void load_row_hint(const unsigned char* __restrict__ tab, long long n_pad, long long s,
                                              unsigned (&w)[Row<D>::W], unsigned long long pol) {
    using R = Row<D>;
#pragma unroll
    for (int p = 0; p < R::N4; ++p) {
        uint4 v = ld_stream16_hint(tab + (size_t)p * 16u * (size_t)n_pad + (size_t)s * 16u, pol);
        w[4 * p + 0] = v.x; w[4 * p + 1] = v.y; w[4 * p + 2] = v.z; w[4 * p + 3] = v.w;
    }
    if constexpr (R::N2 != 0) {
        uint2 v = ld_stream8_hint(tab + (size_t)R::N4 * 16u * (size_t)n_pad + (size_t)s * 8u, pol);
        w[4 * R::N4 + 0] = v.x; w[4 * R::N4 + 1] = v.y;
    }
    if constexpr (R::N1 != 0) {
        w[R::W - 1] = ld_stream4_hint(tab + ((size_t)R::N4 * 16u + (size_t)R::N2 * 8u) * (size_t)n_pad + (size_t)s * 4u, pol);
    }
}

// Load the row of local state `s` from the table that starts at `tab`.
template <int D>
__device__ __forceinline__ void load_row(const unsigned char* __restrict__ tab, long long n_pad, long long s,
                                         unsigned (&w)[Row<D>::W]) {
    using R = Row<D>;
#pragma unroll
    for (int p = 0; p < R::N4; ++p) {
        uint4 v = ld_stream16(tab + (size_t)p * 16u * (size_t)n_pad + (size_t)s * 16u);
        w[4 * p + 0] = v.x; w[4 * p + 1] = v.y; w[4 * p + 2] = v.z; w[4 * p + 3] = v.w;
    }
    if constexpr (R::N2 != 0) {
        uint2 v = ld_stream8(tab + (size_t)R::N4 * 16u * (size_t)n_pad + (size_t)s * 8u);
        w[4 * R::N4 + 0] = v.x; w[4 * R::N4 + 1] = v.y;
    }
    if constexpr (R::N1 != 0) {
        w[R::W - 1] = ld_stream4(tab + ((size_t)R::N4 * 16u + (size_t)R::N2 * 8u) * (size_t)n_pad + (size_t)s * 4u);
    }
}

template <int D>
__device__ __forceinline__ void store_row(unsigned char* __restrict__ tab, long long n_pad, long long s,
                                          const unsigned (&w)[Row<D>::W]) {
    using R = Row<D>;
#pragma unroll
    for (int p = 0; p < R::N4; ++p) {
        st_stream16(tab + (size_t)p * 16u * (size_t)n_pad + (size_t)s * 16u,
                    make_uint4(w[4 * p], w[4 * p + 1], w[4 * p + 2], w[4 * p + 3]));
    }
    if constexpr (R::N2 != 0) {
        st_stream8(tab + (size_t)R::N4 * 16u * (size_t)n_pad + (size_t)s * 8u,
                   make_uint2(w[4 * R::N4], w[4 * R::N4 + 1]));
    }
    if constexpr (R::N1 != 0) {
        st_stream4(tab + ((size_t)R::N4 * 16u + (size_t)R::N2 * 8u) * (size_t)n_pad + (size_t)s * 4u, w[R::W - 1]);
    }
}

// ---------------------------------------------------------------------------
// Corner enumeration of the reference.
//   D == 2 : idxs[0..3] = (i0,i1) (i0,i1+1) (i0+1,i1) (i0+1,i1+1)   (:201-209)
//            -> bit of dim d in corner c is (c >> (1-d)) & 1
//   D >= 3 : bit d of c selects i[d] or i[d]+1                       (:602-613, :1030-1041)
// ---------------------------------------------------------------------------
template <int D>
__host__ __device__ constexpr int corner_bit(int c, int d) {
    return D == 2 ? ((c >> (1 - d)) & 1) : ((c >> d) & 1);
}

// Expected next-state value  sum_c w_c * V[idx_c]  with the reference's exact
// arithmetic: w_c = ((((1*f_0)*f_1)...)*f_{D-1}), f_d = bit ? frac_d : 1-frac_d,
// accumulated as ev = fmaf(w_c, V[idx_c], ev) for c = 0 .. 2^D-1 from ev = 0
// (:236-239, :643-646, :1074-1076).  Prefix products are shared between corners
// (same multiplication order per corner, so the same rounding).
__device__ __forceinline__ float ld_nc_ordered(const float* p) {   // volatile: keeps its place among the other gathers
    float r;
    asm volatile("ld.global.nc.f32 %0, [%1];" : "=f"(r) : "l"(p));
    return r;
}

// Explicitly scheduled form of expected_value (same arithmetic, same order): the 2^D gathers are issued in
// groups of G back-to-back loads, group g+1 before the fma chain of group g consumes its values, so a
// warp always has G..2G gathers in flight whatever ptxas would have hoisted (the sweep is latency-bound:
// measured 1.54 / 1.68 / 1.91 ms for 25 / 21 / 19 leading loads in otherwise equal code).  Weight tree
// over the first D-2 dims, the last two factors applied per corner.
template <int D, int G>
__device__ __forceinline__ float expected_value_grouped(const float* __restrict__ V, int base,
                                                        const float (&frac)[D], const int (&stride)[D]) {
    static_assert(D >= 4, "grouped form needs D >= 4");
    constexpr int C = 1 << D, Q = C / 4, NG = C / G;
    static_assert(C % G == 0 && NG >= 1, "G must divide 2^D");
    float pre[Q];
    pre[0] = 1.0f - frac[0];
    pre[1] = frac[0];
#pragma unroll
    for (int d = 1; d < D - 2; ++d) {
        const float g = 1.0f - frac[d];
#pragma unroll
        for (int c = (1 << d) - 1; c >= 0; --c) {
            const float p = pre[c];
            pre[c + (1 << d)] = p * frac[d];
            pre[c] = p * g;
        }
    }
    const float fm = frac[D - 2], gm = 1.0f - fm, fl = frac[D - 1], gl = 1.0f - fl;
    const float* v = V + base;
    float buf[2][G];
    auto off_of = [&](int c) {
        int off = 0;
#pragma unroll
        for (int d = 0; d < D; ++d)
            if (corner_bit<D>(c, d)) off += stride[d];
        return off;
    };
#pragma unroll
    for (int i = 0; i < G; ++i) buf[0][i] = ld_nc_ordered(v + off_of(i));
    float ev = 0.0f;
#pragma unroll
    for (int g = 0; g < NG; ++g) {
        if (g + 1 < NG) {
#pragma unroll
            for (int i = 0; i < G; ++i) buf[(g + 1) & 1][i] = ld_nc_ordered(v + off_of((g + 1) * G + i));
        }
#pragma unroll
        for (int i = 0; i < G; ++i) {
            const int c = g * G + i;
            const float w = (pre[c & (Q - 1)] * (((c >> (D - 2)) & 1) ? fm : gm)) * ((c >> (D - 1)) ? fl : gl);
            ev = fmaf(w, buf[g & 1][i], ev);
        }
    }
    return ev;
}

// CG = true: gathers bypass the L1 (ld.global.cg) — the persistent multi-sweep kernel reads values other
// SMs wrote one grid barrier ago, and the L1 is not coherent.
template <bool CG>
__device__ __forceinline__ float ld_v(const float* p) {
    if constexpr (CG) return __ldcg(p);
    else return *p;
}

template <int D, bool KEEP = false, int LV = 0, bool CG = false>
__device__ __forceinline__ float expected_value(const float* __restrict__ V, int base,
                                                const float (&frac)[D], const int (&stride)[D],
                                                unsigned long long keep_pol = 0ull) {
    constexpr int C = 1 << D;
    if constexpr (LV == 1 && D >= 4) {
        // Register-lean form: prefix products over the first D-2 dims only (2^(D-2) registers instead of
        // 2^(D-1)); the factors of dims D-2 and D-1 are applied per corner, in the same left-to-right
        // order ((pre * f_{D-2}) * f_{D-1}) — one more multiply per corner, identical rounding.
        constexpr int Q = C / 4;
        float pre[Q];
        pre[0] = 1.0f - frac[0];
        pre[1] = frac[0];
#pragma unroll
        for (int d = 1; d < D - 2; ++d) {
            const float g = 1.0f - frac[d];
#pragma unroll
            for (int c = (1 << d) - 1; c >= 0; --c) {
                const float p = pre[c];
                pre[c + (1 << d)] = p * frac[d];
                pre[c] = p * g;
            }
        }
        const float fm = frac[D - 2], gm = 1.0f - fm, fl = frac[D - 1], gl = 1.0f - fl;
        const float* v = V + base;
        float ev = 0.0f;
#pragma unroll
        for (int c = 0; c < C; ++c) {
            int off = 0;
#pragma unroll
            for (int d = 0; d < D; ++d)
                if (corner_bit<D>(c, d)) off += stride[d];
            float x;
            if constexpr (KEEP) x = ld_keep4(v + off, keep_pol);
            else x = v[off];
            const float w = (pre[c & (Q - 1)] * (((c >> (D - 2)) & 1) ? fm : gm)) * ((c >> (D - 1)) ? fl : gl);
            ev = fmaf(w, x, ev);
        }
        return ev;
    } else
    if constexpr (D == 1) {
        const float* v = V + base;
        float ev = fmaf(1.0f - frac[0], ld_v<CG>(v), 0.0f);
        return fmaf(frac[0], ld_v<CG>(v + stride[0]), ev);
    } else if constexpr (D == 2) {
        const float g0 = 1.0f - frac[0], g1 = 1.0f - frac[1];
        const float* v = V + base;
        const float v00 = ld_v<CG>(v), v01 = ld_v<CG>(v + stride[1]), v10 = ld_v<CG>(v + stride[0]),
                    v11 = ld_v<CG>(v + stride[0] + stride[1]);
        float ev = 0.0f;
        ev = fmaf(g0 * g1, v00, ev);
        ev = fmaf(g0 * frac[1], v01, ev);
        ev = fmaf(frac[0] * g1, v10, ev);
        ev = fmaf(frac[0] * frac[1], v11, ev);
        return ev;
    } else {
        // weights over the first D-1 dims (2^(D-1) prefix products), last dim applied on the fly
        constexpr int H = C / 2;
        float pre[H];
        pre[0] = 1.0f - frac[0];
        pre[1] = frac[0];
#pragma unroll
        for (int d = 1; d < D - 1; ++d) {
            const float g = 1.0f - frac[d];
#pragma unroll
            for (int c = (1 << d) - 1; c >= 0; --c) {
                const float p = pre[c];
                pre[c + (1 << d)] = p * frac[d];
                pre[c] = p * g;
            }
        }
        const float gl = 1.0f - frac[D - 1];
        const float* v = V + base;
        float val[C];
#pragma unroll
        for (int c = 0; c < C; ++c) {
            int off = 0;
#pragma unroll
            for (int d = 0; d < D; ++d)
                if (corner_bit<D>(c, d)) off += stride[d];
            if constexpr (KEEP) val[c] = ld_keep4(v + off, keep_pol);
            else val[c] = ld_v<CG>(v + off);
        }
        float ev = 0.0f;
#pragma unroll
        for (int c = 0; c < H; ++c) ev = fmaf(pre[c] * gl, val[c], ev);
#pragma unroll
        for (int c = 0; c < H; ++c) ev = fmaf(pre[c] * frac[D - 1], val[c + H], ev);
        return ev;
    }
}

__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

// How regular are the rows of the current policy along the fast-stored dimension?  A group of K
// consecutive states is regular when every live state has base_j - j == A with A % K in {0, K-1}
// (the window condition of the x-line sweep, xline_sweep_src.cuh).  Called by all threads of a
// block whose thread index == local state index modulo 32 (groups never straddle a warp);
// counters: [0] pairs, [1] regular pairs, [2] quads, [3] regular quads.
__device__ __forceinline__ void count_regular_groups(int base, bool in, unsigned long long* counters) {
    if (counters == nullptr) return;
    // Only the FRACTION matters: on large grids every 4th block is counted, reduced in shared memory,
    // and adds 4 global atomics (an atomic per warp cost 8 ms on K5: 8 M same-address atomics).
    if (gridDim.x > 1024 && (blockIdx.x & 3) != 0) return;
    __shared__ unsigned s_cnt[4];
    if (threadIdx.x < 4) s_cnt[threadIdx.x] = 0;
    __syncthreads();
    const unsigned full = 0xffffffffu;
    const int lane = threadIdx.x & 31;
    const bool live = base >= 0;
    const unsigned livem = __ballot_sync(full, live);
#pragma unroll
    for (int K = 2; K <= 4; K += 2) {
        const int j = lane % K;
        const unsigned gmask = ((1u << K) - 1u) << (lane - j);
        const unsigned lm = livem & gmask;
        const int t = base - j;
        const int A = __shfl_sync(full, t, lm ? __ffs(lm) - 1 : lane);
        const unsigned okm = __ballot_sync(full, !live || t == A) & gmask;
        const int m = A & (K - 1);
        const bool regular = lm == 0 || (okm == gmask && (m == 0 || m == K - 1));
        const unsigned heads = __ballot_sync(full, in && j == 0);
        const unsigned regs = __ballot_sync(full, in && j == 0 && regular);
        if (lane == 0 && heads) {
            atomicAdd(&s_cnt[K - 2], (unsigned)__popc(heads));
            atomicAdd(&s_cnt[K - 1], (unsigned)__popc(regs));
        }
    }
    __syncthreads();
    if (threadIdx.x < 4 && s_cnt[threadIdx.x]) atomicAdd(counters + threadIdx.x, (unsigned long long)s_cnt[threadIdx.x]);
}

// ---------------------------------------------------------------------------
// Evaluation sweep: one Jacobi Bellman backup of every local state with the
// residual fused in (replaces policy_eval_kernel* + the max_abs_diff
// ReductionKernel, src/cuda_policy_iteration.py:212-242, :616-649, :1044-1079,
// :164-172).  Launched back to back; each launch reads the sweep counter from
// the control block, so a CUDA graph of identical nodes runs a whole sync
// interval.
// ---------------------------------------------------------------------------
struct EvalParams {
    const unsigned char* rows;  // compacted rows of the current policy (n_pad states)
    float* V0;                  // ping
    float* V1;                  // pong  (both full length n_states)
    Ctl* ctl;
    float* partial;             // per-block residual maxima (written on check sweeps only)
    long long n_local;
    long long n_pad;
    long long s_begin;  // first global state of this rank
    float gamma;
    int j;      // position of this launch inside its batch: sweep index = ctl->base + j
    int check;  // 1 if the host will examine the residual of this sweep (sync point, :325)
    int lookahead;  // blocks ahead whose rows are prefetched into L2 (0 = off)
    int stride[kMaxDims];
    PeerOut peers;  // sharded runs with the fused exchange: where else new values go (n = 0: nowhere)
};

// TMA bulk prefetch of `bytes` (multiple of 16) starting at p into L2.
__device__ __forceinline__ void prefetch_l2_bulk(const void* p, unsigned bytes) {
    asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(p), "r"(bytes) : "memory");
}
__device__ __forceinline__ void prefetch_l2_bulk_hint(const void* p, unsigned bytes, unsigned long long pol) {
    asm volatile("cp.async.bulk.prefetch.L2.global.L2::cache_hint [%0], %1, %2;" ::"l"(p), "r"(bytes), "l"(pol) : "memory");
}

// Blocks are scheduled in index order, so at any moment all SMs work in one
// neighbourhood of the state space and share its V window in L2 (a persistent kernel
// with one contiguous chunk per block was tried: it doubled DRAM traffic, L2 hit rate
// 55 % -> 22 %).  What in-order scheduling leaves exposed is the DRAM latency of the
// row stream at the start of every block; one thread per block therefore issues a TMA
// bulk prefetch into L2 of the row planes (and the old values) that the block
// `p.lookahead` positions later will read.
// VAR (tuning variants, selected by DPB200_EVAL_VARIANT; all bit-identical):
//   bit 0: L2 evict-first policy on the row stream (loads and the TMA prefetch)
//   bit 1: L2 evict-last policy on the V gathers
//   bits 2-4: minimum resident blocks per SM forced through __launch_bounds__:
//             0 -> unspecified (compiler heuristic), 1 -> 1, 2 -> 3, 3 -> 4, 4 -> 5, 5 -> 6, 6 -> 8
__host__ __device__ constexpr int eval_variant_minb(int var) {
    constexpr int t[8] = {0, 1, 3, 4, 5, 6, 8, 0};
    return t[(var >> 2) & 7];
}
template <int D, int VAR = 0>
__global__ void __launch_bounds__(kBlock, eval_variant_minb(VAR)) eval_sweep_kernel(const EvalParams p) {
    constexpr bool ROW_EF = (VAR & 1) != 0, V_KEEP = (VAR & 2) != 0;
    constexpr int LEAN = (VAR >> 5) & 1;   // bit 5: register-lean weight tree (expected_value LV = 1)
    // bits 6-8: explicitly scheduled gathers in groups of 8 / 16 / 32 / 4 / 2 (expected_value_grouped)
    constexpr int kGroupOf[8] = {0, 8, 16, 32, 4, 2, 0, 0};
    constexpr int GROUP = kGroupOf[(VAR >> 6) & 7];
    const Ctl* __restrict__ ctl = p.ctl;
    if (ctl->done) return;
    const int par = (ctl->base + p.j + ctl->parity0) & 1;
    const float* __restrict__ Vin = par ? p.V1 : p.V0;
    float* __restrict__ Vout = par ? p.V0 : p.V1;

    if (threadIdx.x == 0 && p.lookahead > 0) {
        const long long s_pf = ((long long)blockIdx.x + p.lookahead) * kBlock;
        if (s_pf < p.n_local) {
            using R = Row<D>;
            const long long left = p.n_pad - s_pf;
            const unsigned n = (unsigned)(left < kBlock ? left : kBlock);
            if constexpr (ROW_EF) {
                const unsigned long long pol = l2_policy_evict_first();
#pragma unroll
                for (int q = 0; q < R::N4; ++q)
                    prefetch_l2_bulk_hint(p.rows + (size_t)q * 16u * (size_t)p.n_pad + (size_t)s_pf * 16u, n * 16u, pol);
                if constexpr (R::N2 != 0)
                    prefetch_l2_bulk_hint(p.rows + (size_t)R::N4 * 16u * (size_t)p.n_pad + (size_t)s_pf * 8u, n * 8u, pol);
            } else {
#pragma unroll
                for (int q = 0; q < R::N4; ++q)
                    prefetch_l2_bulk(p.rows + (size_t)q * 16u * (size_t)p.n_pad + (size_t)s_pf * 16u, n * 16u);
                if constexpr (R::N2 != 0)
                    prefetch_l2_bulk(p.rows + (size_t)R::N4 * 16u * (size_t)p.n_pad + (size_t)s_pf * 8u, n * 8u);
            }
        }
    }

    const long long s = (long long)blockIdx.x * kBlock + threadIdx.x;
    float res = 0.0f;
    if (s < p.n_local) {
        unsigned w[Row<D>::W];
        if constexpr (ROW_EF) load_row_hint<D>(p.rows, p.n_pad, s, w, l2_policy_evict_first());
        else load_row<D>(p.rows, p.n_pad, s, w);
        const int base = (int)w[0];
        const float vold = Vin[p.s_begin + s];
        float vnew;
        if (base == PI_ROW_ABSORBING) {
            vnew = vold;  // :221 / :625 / :1053
        } else {
            float ev = 0.0f;
            if (base >= 0) {
                float frac[D];
                int stride[D];
#pragma unroll
                for (int d = 0; d < D; ++d) { frac[d] = __uint_as_float(w[1 + d]); stride[d] = p.stride[d]; }
                if constexpr (GROUP != 0 && D >= 4) ev = expected_value_grouped<D, (GROUP < (1 << D) ? GROUP : (1 << D))>(Vin, base, frac, stride);
                else if constexpr (V_KEEP) ev = expected_value<D, true, LEAN>(Vin, base, frac, stride, l2_policy_evict_last());
                else ev = expected_value<D, false, LEAN>(Vin, base, frac, stride);
            }
            vnew = fmaf(p.gamma, ev, __uint_as_float(w[D + 1]));  // reward + gamma*ev contracts to one FMA
        }
        Vout[p.s_begin + s] = vnew;
        if (p.peers.n) store_peers(p.peers, par != 0, p.s_begin + s, vnew);
        res = fabsf(vnew - vold);
    }
    if (!p.check) return;  // the reference reads the residual only at sync points (:325-326)

    // block residual -> partial[blockIdx]; reduced by eval_reduce_kernel (no atomics on the sweep path)
    __shared__ float s_red[kBlock / 32];
    res = warp_max(res);
    if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = res;
    __syncthreads();
    if (threadIdx.x < 32) {
        float r = threadIdx.x < kBlock / 32 ? s_red[threadIdx.x] : 0.0f;
        r = warp_max(r);
        if (threadIdx.x == 0) p.partial[blockIdx.x] = r;
    }
}

// ---------------------------------------------------------------------------
// Persistent multi-sweep evaluation for grids that fit the chip: ONE cooperative launch runs a whole
// batch of sweeps (up to a sync interval of policy_evaluation(), src/cuda_policy_iteration.py:300-336).
// Small grids (K1 Pendulum 200^2, K2 Continuous Mountain Car 400^2) are launch-bound in the per-sweep
// form: 2.4 us per sweep of which the Bellman backups are a fraction.  Here every thread keeps the rows
// of its (up to SPT) states in registers for the whole batch, V lives in L2 (gathers bypass the
// non-coherent L1), sweeps are separated by a grid barrier (one release-arrive + acquire-spin per block on a
// monotonic counter) instead of a kernel boundary, and the residual reduction + bookkeeping of
// eval_reduce_kernel is done by the last block to finish.  Same arithmetic, same order, same sweep counts.
// ---------------------------------------------------------------------------
constexpr int kPBlock = 512;

struct PersistParams {
    const unsigned char* rows;
    float* V0;
    float* V1;
    Ctl* ctl;
    float* partial;      // [gridDim.x]
    unsigned* bar;       // [0] barrier arrivals, [1] finish tickets — zeroed before every launch
    long long n_local;
    long long n_pad;
    float gamma;
    float theta;
    int k;               // sweeps in this launch
    int has_check;       // reduce the residual of the last sweep
    int decide;          // ... and apply delta < theta (kBatchDecide)
    int stride[kMaxDims];
};

__device__ __forceinline__ unsigned ld_acquire_u32(const unsigned* p) {
    unsigned v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}

// All blocks are co-resident (cooperative launch).  `target` counts arrivals expected so far.
__device__ __forceinline__ void grid_barrier(unsigned* bar, unsigned& target) {
    __syncthreads();
    if (threadIdx.x == 0) {
        target += gridDim.x;
        __threadfence();   // this block's V stores are visible before its arrival is
        atomicAdd(bar, 1u);
        while (ld_acquire_u32(bar) < target) { }
    }
    __syncthreads();
}

template <int D, int SPT>
__global__ void __launch_bounds__(kPBlock) eval_persistent_kernel(const PersistParams p) {
    Ctl* ctl = p.ctl;
    if (ctl->done) return;   // written by an earlier launch: every block sees the same value
    const int par0 = (ctl->base + ctl->parity0) & 1;
    const long long tid = (long long)blockIdx.x * kPBlock + threadIdx.x;
    const long long nthreads = (long long)gridDim.x * kPBlock;

    unsigned w[SPT][Row<D>::W];
    float vcur[SPT];
    bool in[SPT];
    int stride[D];
#pragma unroll
    for (int d = 0; d < D; ++d) stride[d] = p.stride[d];
#pragma unroll
    for (int i = 0; i < SPT; ++i) {
        const long long s = tid + i * nthreads;
        in[i] = s < p.n_local;
        vcur[i] = 0.0f;
        if (in[i]) {
            load_row<D>(p.rows, p.n_pad, s, w[i]);
            vcur[i] = __ldcg((par0 ? p.V1 : p.V0) + s);
        }
    }

    unsigned target = 0;
    float res = 0.0f;
    for (int j = 0; j < p.k; ++j) {
        const int par = (par0 + j) & 1;
        const float* Vin = par ? p.V1 : p.V0;
        float* Vout = par ? p.V0 : p.V1;
        const bool last = j == p.k - 1;
#pragma unroll
        for (int i = 0; i < SPT; ++i) {
            if (!in[i]) continue;
            const int base = (int)w[i][0];
            const float vold = vcur[i];
            float vnew;
            if (base == PI_ROW_ABSORBING) {
                vnew = vold;
            } else {
                float ev = 0.0f;
                if (base >= 0) {
                    float frac[D];
#pragma unroll
                    for (int d = 0; d < D; ++d) frac[d] = __uint_as_float(w[i][1 + d]);
                    ev = expected_value<D, false, 0, true>(Vin, base, frac, stride);
                }
                vnew = fmaf(p.gamma, ev, __uint_as_float(w[i][D + 1]));
            }
            __stcg(Vout + tid + i * nthreads, vnew);
            vcur[i] = vnew;
            if (last) res = fmaxf(res, fabsf(vnew - vold));
        }
        if (!last) grid_barrier(p.bar, target);
    }

    // residual of the last sweep -> partial[block]; the last block to finish reduces and keeps the books
    __shared__ float s_red[kPBlock / 32];
    __shared__ int s_is_last;
    if (p.has_check) {
        res = warp_max(res);
        if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = res;
        __syncthreads();
        if (threadIdx.x < 32) {
            float r = threadIdx.x < kPBlock / 32 ? s_red[threadIdx.x] : 0.0f;
            r = warp_max(r);
            if (threadIdx.x == 0) __stcg(p.partial + blockIdx.x, r);
        }
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        s_is_last = atomicAdd(p.bar + 1, 1u) == gridDim.x - 1;
    }
    __syncthreads();
    if (!s_is_last) return;
    __threadfence();
    float r = 0.0f;
    if (p.has_check) {
        for (int b = threadIdx.x; b < (int)gridDim.x; b += kPBlock) r = fmaxf(r, __ldcg(p.partial + b));
        r = warp_max(r);
        __syncthreads();
        if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = r;
        __syncthreads();
        if (threadIdx.x < 32) {
            r = threadIdx.x < kPBlock / 32 ? s_red[threadIdx.x] : 0.0f;
            r = warp_max(r);
        }
    }
    if (threadIdx.x == 0) {   // == eval_reduce_kernel
        ctl->base += p.k;
        if (p.has_check) {
            ctl->last_delta = r;
            if (p.decide) {
                ctl->check_delta = r;
                if (r < p.theta) { ctl->done = 1; ctl->conv_sweep = ctl->base - 1; }
            }
        }
    }
}

// ---------------------------------------------------------------------------
// Evaluation sweep, TWO consecutive states per thread along the fastest-stored
// dimension (logical dimension F, istride[F] == 1).
//
// When the two states' successor cells are neighbours along F (base_1 == base_0 + 1
// — the common case once the layout probe has put a well-behaved dimension
// fastest), the 2^D corners of both states live in 2^(D-1) three-element windows
// V[a], V[a+1], V[a+2]: state 0 uses (a, a+1), state 1 uses (a+1, a+2).  Each window
// is fetched with two aligned 64-bit loads, so the pair needs 2^D 64-bit requests
// instead of 2*2^D 32-bit ones, and the L1 data-pipe wavefronts (the binding unit
// of the scalar kernel, see DESIGN.md §5) drop by almost 2x.  Rows of the two
// states are one 256-bit load per 16-byte plane.  The fma chain of each state is
// still evaluated in ascending corner order with individually rounded weights, so
// the result is bit-identical to eval_sweep_kernel.  Any other pair (sentinel rows,
// clamped / non-adjacent successors) takes the scalar path.
// ---------------------------------------------------------------------------
__device__ __forceinline__ void ld_stream32(const void* p, unsigned (&r)[8]) {
    asm volatile("ld.global.nc.L1::no_allocate.v8.u32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
                 : "l"(p));
}

// rows of local states s0 (even) and s0 + 1
template <int D>
__device__ __forceinline__ void load_row2(const unsigned char* __restrict__ tab, long long n_pad, long long s0,
                                          unsigned (&w0)[Row<D>::W], unsigned (&w1)[Row<D>::W]) {
    using R = Row<D>;
#pragma unroll
    for (int p = 0; p < R::N4; ++p) {
        unsigned r[8];
        ld_stream32(tab + (size_t)p * 16u * (size_t)n_pad + (size_t)s0 * 16u, r);
#pragma unroll
        for (int k = 0; k < 4; ++k) { w0[4 * p + k] = r[k]; w1[4 * p + k] = r[4 + k]; }
    }
    if constexpr (R::N2 != 0) {
        uint4 v = ld_stream16(tab + (size_t)R::N4 * 16u * (size_t)n_pad + (size_t)s0 * 8u);
        w0[4 * R::N4] = v.x; w0[4 * R::N4 + 1] = v.y; w1[4 * R::N4] = v.z; w1[4 * R::N4 + 1] = v.w;
    }
    if constexpr (R::N1 != 0) {
        uint2 v = ld_stream8(tab + ((size_t)R::N4 * 16u + (size_t)R::N2 * 8u) * (size_t)n_pad + (size_t)s0 * 4u);
        w0[R::W - 1] = v.x; w1[R::W - 1] = v.y;
    }
}

// bit position of logical dimension d inside a corner number (see corner_bit)
template <int D>
__host__ __device__ constexpr int corner_pos(int d) { return D == 2 ? 1 - d : d; }

// prefix products over dims 0..D-2 (2^(D-1) values), reference multiplication order
template <int D>
__device__ __forceinline__ void prefix_weights(const float (&frac)[D], float (&pre)[(1 << D) / 2]) {
    if constexpr (D >= 3) {
        pre[0] = 1.0f - frac[0];
        pre[1] = frac[0];
#pragma unroll
        for (int d = 1; d < D - 1; ++d) {
            const float g = 1.0f - frac[d];
#pragma unroll
            for (int c = (1 << d) - 1; c >= 0; --c) {
                const float q = pre[c];
                pre[c + (1 << d)] = q * frac[d];
                pre[c] = q * g;
            }
        }
    } else {
        pre[0] = 0.0f;  // unused for D <= 2
    }
}
template <int D>
__device__ __forceinline__ float corner_weight(const float (&frac)[D], const float (&pre)[(1 << D) / 2], int c) {
    if constexpr (D == 1) {
        return c ? frac[0] : 1.0f - frac[0];
    } else if constexpr (D == 2) {
        const float a = corner_bit<2>(c, 0) ? frac[0] : 1.0f - frac[0];
        const float b = corner_bit<2>(c, 1) ? frac[1] : 1.0f - frac[1];
        return a * b;
    } else {
        constexpr int H = (1 << D) / 2;
        return pre[c & (H - 1)] * ((c & H) ? frac[D - 1] : 1.0f - frac[D - 1]);
    }
}

template <int D, int F>
__global__ void __launch_bounds__(kBlock) eval_sweep_pair_kernel(const EvalParams p) {
    constexpr int W = Row<D>::W;
    constexpr int C = 1 << D;
    constexpr int P = corner_pos<D>(F);     // bit position of the fast dimension in a corner number
    constexpr int NLO = 1 << P;             // row-combos below the fast bit
    constexpr int NHI = C >> (P + 1);       // row-combos above it
    const Ctl* __restrict__ ctl = p.ctl;
    if (ctl->done) return;
    const int par = (ctl->base + p.j + ctl->parity0) & 1;
    const float* __restrict__ Vin = par ? p.V1 : p.V0;
    float* __restrict__ Vout = par ? p.V0 : p.V1;

    const long long s0 = 2 * ((long long)blockIdx.x * kBlock + threadIdx.x);
    float res = 0.0f;
    if (s0 < p.n_local) {
        const bool has1 = s0 + 1 < p.n_local;
        unsigned w0[W], w1[W];
        load_row2<D>(p.rows, p.n_pad, s0, w0, w1);
        const int b0 = (int)w0[0], b1 = (int)w1[0];
        const long long g0 = p.s_begin + s0;
        float vold0, vold1 = 0.0f;
        if ((g0 & 1) == 0) {
            const float2 t = *reinterpret_cast<const float2*>(Vin + g0);  // V buffers are padded, s0+1 is readable
            vold0 = t.x; vold1 = t.y;
        } else {
            vold0 = Vin[g0];
            if (has1) vold1 = Vin[g0 + 1];
        }
        float vnew0, vnew1 = 0.0f;
        int stride[D];
#pragma unroll
        for (int d = 0; d < D; ++d) stride[d] = p.stride[d];

        // Effective bases: a sentinel row (terminated / absorbing / padding) borrows its partner's
        // cell so that its (discarded) loads stay in range; delta = distance between the two
        // successor cells along the fast dimension.  delta == 1: neighbours; delta == 0: same cell
        // (clamped at a grid edge, or one row is a sentinel).  Anything else -> scalar path.
        const bool sen0 = b0 < 0, sen1 = !has1 || b1 < 0;
        const int e0 = sen0 ? (sen1 ? 0 : b1) : b0;
        const int e1 = sen1 ? e0 : b1;
        const int delta = e1 - e0;
        if (delta == 0 || delta == 1) {
            float f0[D], f1[D];
#pragma unroll
            for (int d = 0; d < D; ++d) { f0[d] = __uint_as_float(w0[1 + d]); f1[d] = __uint_as_float(w1[1 + d]); }
            float pre0[C / 2], pre1[C / 2];
            prefix_weights<D>(f0, pre0);
            prefix_weights<D>(f1, pre1);
            float ev0 = 0.0f, ev1 = 0.0f;
#pragma unroll
            for (int hi = 0; hi < NHI; ++hi) {
                float x[NLO][3];
#pragma unroll
                for (int lo = 0; lo < NLO; ++lo) {
                    const int c = (hi << (P + 1)) | lo;  // corner with the fast bit clear
                    int off = 0;
#pragma unroll
                    for (int d = 0; d < D; ++d)
                        if (d != F && corner_bit<D>(c, d)) off += stride[d];
                    const int a = e0 + off;
                    const float2* q = reinterpret_cast<const float2*>(Vin + (a & ~1));
                    const float2 r01 = q[0], r23 = q[1];
                    const bool odd = a & 1;
                    x[lo][0] = odd ? r01.y : r01.x;
                    x[lo][1] = odd ? r23.x : r01.y;
                    x[lo][2] = odd ? r23.y : r23.x;
                }
#pragma unroll
                for (int fb = 0; fb < 2; ++fb) {
#pragma unroll
                    for (int lo = 0; lo < NLO; ++lo) {
                        const int c = (hi << (P + 1)) | (fb << P) | lo;
                        ev0 = fmaf(corner_weight<D>(f0, pre0, c), x[lo][fb], ev0);
                        ev1 = fmaf(corner_weight<D>(f1, pre1, c), delta ? x[lo][fb + 1] : x[lo][fb], ev1);
                    }
                }
            }
            // sentinel rows: terminated -> sum := 0 (:231-232); absorbing -> new_V := V (:221)
            vnew0 = b0 == PI_ROW_ABSORBING ? vold0 : fmaf(p.gamma, sen0 ? 0.0f : ev0, __uint_as_float(w0[D + 1]));
            vnew1 = b1 == PI_ROW_ABSORBING ? vold1 : fmaf(p.gamma, sen1 ? 0.0f : ev1, __uint_as_float(w1[D + 1]));
        } else {
            // scalar path, one state at a time (identical to eval_sweep_kernel)
            if (b0 == PI_ROW_ABSORBING) {
                vnew0 = vold0;
            } else {
                float ev = 0.0f;
                if (b0 >= 0) {
                    float fr[D];
#pragma unroll
                    for (int d = 0; d < D; ++d) fr[d] = __uint_as_float(w0[1 + d]);
                    ev = expected_value<D>(Vin, b0, fr, stride);
                }
                vnew0 = fmaf(p.gamma, ev, __uint_as_float(w0[D + 1]));
            }
            if (has1) {
                if (b1 == PI_ROW_ABSORBING) {
                    vnew1 = vold1;
                } else {
                    float ev = 0.0f;
                    if (b1 >= 0) {
                        float fr[D];
#pragma unroll
                        for (int d = 0; d < D; ++d) fr[d] = __uint_as_float(w1[1 + d]);
                        ev = expected_value<D>(Vin, b1, fr, stride);
                    }
                    vnew1 = fmaf(p.gamma, ev, __uint_as_float(w1[D + 1]));
                }
            }
        }
        if ((g0 & 1) == 0 && has1) {
            *reinterpret_cast<float2*>(Vout + g0) = make_float2(vnew0, vnew1);
        } else {
            Vout[g0] = vnew0;
            if (has1) Vout[g0 + 1] = vnew1;
        }
        if (p.peers.n) {
            store_peers(p.peers, par != 0, g0, vnew0);
            if (has1) store_peers(p.peers, par != 0, g0 + 1, vnew1);
        }
        res = fabsf(vnew0 - vold0);
        if (has1) res = fmaxf(res, fabsf(vnew1 - vold1));
    }
    if (!p.check) return;
    __shared__ float s_red[kBlock / 32];
    res = warp_max(res);
    if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = res;
    __syncthreads();
    if (threadIdx.x < 32) {
        float r = threadIdx.x < kBlock / 32 ? s_red[threadIdx.x] : 0.0f;
        r = warp_max(r);
        if (threadIdx.x == 0) p.partial[blockIdx.x] = r;
    }
}

// End of a batch of k sweeps: advance the sweep counter; if the last sweep was a
// check sweep, reduce the per-block residuals; if `decide`, apply the sync-point
// test of policy_evaluation (:325-331).  When sharded the residual is all-reduced
// between this kernel (decide = 0) and eval_decide_kernel.
__global__ void __launch_bounds__(1024) eval_reduce_kernel(Ctl* ctl, const float* partial, int n_partial, int k,
                                                          int has_check, int decide, float theta) {
    if (ctl->done) return;
    __shared__ float s_red[32];
    float r = 0.0f;
    if (has_check) {
        for (int i = threadIdx.x; i < n_partial; i += blockDim.x) r = fmaxf(r, partial[i]);
        r = warp_max(r);
        if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = r;
        __syncthreads();
        if (threadIdx.x < 32) {
            r = threadIdx.x < (blockDim.x >> 5) ? s_red[threadIdx.x] : 0.0f;
            r = warp_max(r);
        }
    }
    if (threadIdx.x == 0) {
        ctl->base += k;
        if (has_check) {
            ctl->last_delta = r;
            if (decide) {
                ctl->check_delta = r;
                if (r < theta) { ctl->done = 1; ctl->conv_sweep = ctl->base - 1; }
            }
        }
    }
}

// First level of a two-level reduction of the per-block partials (max of floats / sum of counts): the one-block
// final kernels above read 500 000 partials of a 64 M-state sweep in 204 us; 256 blocks bring that to a few us.
__global__ void __launch_bounds__(256) partial_max_kernel(const float* __restrict__ in, int n, float* __restrict__ out) {
    float r = 0.0f;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) r = fmaxf(r, in[i]);
    __shared__ float s_red[8];
    r = warp_max(r);
    if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = r;
    __syncthreads();
    if (threadIdx.x < 32) {
        r = threadIdx.x < 8 ? s_red[threadIdx.x] : 0.0f;
        r = warp_max(r);
        if (threadIdx.x == 0) out[blockIdx.x] = r;
    }
}
__global__ void __launch_bounds__(256) partial_sum_kernel(const unsigned* __restrict__ in, int n, unsigned* __restrict__ out) {
    unsigned r = 0;   // a block sums at most n / gridDim counts of <= 256 each: no overflow below 2^24 partials per block
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) r += in[i];
    __shared__ unsigned s_red[8];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) r += __shfl_xor_sync(0xffffffffu, r, o);
    if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = r;
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned t = 0;
        for (int i = 0; i < 8; ++i) t += s_red[i];
        out[blockIdx.x] = t;
    }
}

__global__ void eval_decide_kernel(Ctl* ctl, const float* delta_src, float theta) {
    if (ctl->done) return;
    const float d = *delta_src;
    ctl->check_delta = d;
    if (d < theta) {
        ctl->done = 1;
        ctl->conv_sweep = ctl->base - 1;
    }
}

__global__ void eval_begin_kernel(Ctl* ctl, int parity0) {
    ctl->base = 0;
    ctl->parity0 = parity0;
    ctl->done = 0;
    ctl->conv_sweep = -1;
    ctl->last_delta = __int_as_float(0x7f800000);
    ctl->check_delta = __int_as_float(0x7f800000);
}

// ---------------------------------------------------------------------------
// Improvement: per state, Q(s,a) for a = 0..A-1 in order, strict '>' from
// -1e30f with best_a = 0 (lowest index wins ties, NaN never wins), absorbing
// states untouched (replaces policy_improve_kernel*, :244-283, :651-691,
// :1081-1123) — fused with (i) the "policy changed" count that replaces
// old_policy.copy() + cp.all(==) (:340,:354) and (ii) compaction of the
// winning row into the evaluation table.
// ---------------------------------------------------------------------------
struct ImproveParams {
    const unsigned char* table;  // [A] row tables, action stride = W*4*n_pad bytes
    unsigned char* rows;         // out: compacted rows of the new policy
    const float* V;              // current value function (full length)
    int* policy;                 // local policy (n_local)
    unsigned int* partial;       // per-block count of states whose action changed
    unsigned long long* regular; // optional: regularity counters of the new policy's rows (count_regular_groups)
    long long n_local;
    long long n_pad;
    int n_actions;
    float gamma;
    int stride[kMaxDims];
};

template <int D>
__global__ void __launch_bounds__(kBlock) improve_kernel(const ImproveParams p) {
    const long long s = (long long)blockIdx.x * kBlock + threadIdx.x;
    int changed = 0;
    int win_base = PI_ROW_ABSORBING;
    if (s < p.n_local) {
        constexpr int W = Row<D>::W;
        const size_t a_stride = (size_t)W * 4u * (size_t)p.n_pad;
        unsigned best_row[W];
        load_row<D>(p.table, p.n_pad, s, best_row);
        const int old_a = p.policy[s];
        if ((int)best_row[0] != PI_ROW_ABSORBING) {
            int stride[D];
#pragma unroll
            for (int d = 0; d < D; ++d) stride[d] = p.stride[d];
            float max_q = -1.0e30f;
            int best_a = 0;
            unsigned w[W];
#pragma unroll
            for (int k = 0; k < W; ++k) w[k] = best_row[k];
            for (int a = 0; a < p.n_actions; ++a) {
                if (a > 0) load_row<D>(p.table + (size_t)a * a_stride, p.n_pad, s, w);
                const int base = (int)w[0];
                float ev = 0.0f;
                if (base >= 0) {
                    float frac[D];
#pragma unroll
                    for (int d = 0; d < D; ++d) frac[d] = __uint_as_float(w[1 + d]);
                    ev = expected_value<D>(p.V, base, frac, stride);
                }
                const float q = fmaf(p.gamma, ev, __uint_as_float(w[D + 1]));
                if (q > max_q) {
                    max_q = q;
                    best_a = a;
#pragma unroll
                    for (int k = 0; k < W; ++k) best_row[k] = w[k];
                }
            }
            p.policy[s] = best_a;
            changed = (best_a != old_a);
        }
        store_row<D>(p.rows, p.n_pad, s, best_row);
        win_base = (int)best_row[0];
    }
    count_regular_groups(win_base, s < p.n_local, p.regular);
    const unsigned m = __ballot_sync(0xffffffffu, changed);
    __shared__ int s_cnt;
    if (threadIdx.x == 0) s_cnt = 0;
    __syncthreads();
    if ((threadIdx.x & 31) == 0 && m) atomicAdd(&s_cnt, __popc(m));
    __syncthreads();
    if (threadIdx.x == 0) p.partial[blockIdx.x] = (unsigned)s_cnt;
}

__global__ void __launch_bounds__(1024) count_reduce_kernel(Ctl* ctl, const unsigned int* partial, int n_partial) {
    __shared__ unsigned long long s_red[32];
    unsigned long long r = 0;
    for (int i = threadIdx.x; i < n_partial; i += blockDim.x) r += partial[i];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) r += __shfl_xor_sync(0xffffffffu, r, o);
    if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = r;
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned long long t = 0;
        for (int i = 0; i < (int)(blockDim.x >> 5); ++i) t += s_red[i];
        ctl->changed = t;
    }
}

// rows[s] = table[policy[s]][s]  (after pi_upload_policy and at start-up)
template <int D>
__global__ void __launch_bounds__(kBlock) compact_rows_kernel(const unsigned char* table, unsigned char* rows,
                                                              const int* policy, long long n_local,
                                                              long long n_pad, unsigned long long* regular, long long s_first = 0) {
    // states [s_first, n_local): s_first a multiple of the warp size (the regularity counters look at aligned groups)
    const long long s = s_first + (long long)blockIdx.x * kBlock + threadIdx.x;
    int base = PI_ROW_ABSORBING;
    if (s < n_local) {
        constexpr int W = Row<D>::W;
        unsigned w[W];
        load_row<D>(table + (size_t)policy[s] * ((size_t)W * 4u * (size_t)n_pad), n_pad, s, w);
        store_row<D>(rows, n_pad, s, w);
        base = (int)w[0];
    }
    count_regular_groups(base, s < n_local, regular);
}

// Expand compact rows to the reference's corner form (parity checks only).
// States are addressed by REFERENCE flat index; indices are converted back to
// reference flat indices.  term: 0 live, 1 terminated, 2 absorbing, 255 not in this shard.
template <int D>
__global__ void expand_rows_kernel(const unsigned char* table, long long n_pad, long long s_ref0, long long count,
                                   GridDesc g, long long s_begin_int, long long n_local, int* idx, float* wgt,
                                   float* reward, unsigned char* term) {
    const long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= count) return;
    constexpr int W = Row<D>::W;
    constexpr int C = 1 << D;
    const long long loc = ref_to_internal(g, s_ref0 + k) - s_begin_int;
    if (loc < 0 || loc >= n_local) {
        if (term) term[k] = 255;
        return;
    }
    unsigned w[W];
    load_row<D>(table, n_pad, loc, w);
    const int base = (int)w[0];
    const int base_ref = base >= 0 ? (int)internal_to_ref(g, base) : base;
    if (reward) reward[k] = __uint_as_float(w[D + 1]);
    if (term) term[k] = base == PI_ROW_TERMINATED ? 1 : (base == PI_ROW_ABSORBING ? 2 : 0);
    for (int c = 0; c < C; ++c) {
        int off = 0;
        float wc = 1.0f;
#pragma unroll
        for (int d = 0; d < D; ++d) {
            const int bit = corner_bit<D>(c, d);
            const float f = __uint_as_float(w[1 + d]);
            off += bit * g.stride[d];
            wc *= bit ? f : (1.0f - f);
        }
        if (idx) idx[k * C + c] = base >= 0 ? base_ref + off : base;
        if (wgt) wgt[k * C + c] = base >= 0 ? wc : 0.0f;
    }
}

// Pair shadow of V for the JIT sweep's GP_PAIRV mode: P[i] = (V[i], V[i+1]) (the last pair's second half is never read).
__global__ void make_pairs_kernel(const float* __restrict__ V, float2* __restrict__ P, long long n) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) P[i] = make_float2(V[i], i + 1 < n ? V[i + 1] : 0.0f);
}

// V[s] = value where mask (reference order) is set; V buffers are in internal order.
__global__ void fill_masked_kernel(GridDesc g, float* V0, float* V1, const unsigned char* mask_ref, long long n,
                                   float value) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n && mask_ref[internal_to_ref(g, i)]) {
        if (V0) V0[i] = value;
        if (V1) V1[i] = value;
    }
}

// out[k] = ref_full[ref index of internal state s_begin + k]   (reference order -> internal slice)
template <typename T>
__global__ void to_internal_kernel(GridDesc g, const T* __restrict__ ref_full, T* __restrict__ out,
                                   long long s_begin, long long n) {
    const long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (k < n) out[k] = ref_full[internal_to_ref(g, s_begin + k)];
}
// ref_out[s_ref] = in_full[internal index of s_ref]            (internal order -> reference order)
template <typename T>
__global__ void to_reference_kernel(GridDesc g, const T* __restrict__ in_full, T* __restrict__ ref_out, long long n) {
    const long long s = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (s < n) ref_out[s] = in_full[ref_to_internal(g, s)];
}

// Layout probe: average number of distinct 128-byte lines the 32 lanes of a warp
// touch when they gather V[base] (rows of one action, `n` consecutive internal states).
__global__ void gather_lines_kernel(const unsigned char* table, int first_plane_bytes, long long n,
                                    unsigned long long* lines, unsigned long long* warps) {
    const long long s = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    int base = -1;
    if (s < n) base = *reinterpret_cast<const int*>(table + (size_t)s * first_plane_bytes);
    const unsigned active = __ballot_sync(0xffffffffu, base >= 0);
    if (base >= 0) {
        const unsigned same = __match_any_sync(active, base >> 5);
        const bool leader = (__ffs(same) - 1) == (int)(threadIdx.x & 31);
        const unsigned leaders = __ballot_sync(active, leader);
        if ((__ffs(active) - 1) == (int)(threadIdx.x & 31)) {
            atomicAdd(lines, (unsigned long long)__popc(leaders));
            atomicAdd(warps, 1ull);
        }
    }
}

// ---------------------------------------------------------------------------
// x-line sweep support (the sweep itself is JIT-compiled from xline_sweep_src.cuh).
// Tile order: the non-fast storage positions k = 0..D-2 are cut into tiles of T_k nodes;
// tiles are enumerated lexicographically (position 0 slowest), the x-lines of a tile
// lexicographically inside it, the S states of an x-line last.
// ---------------------------------------------------------------------------
struct TileGeo {
    int n_pos;               // D - 1
    int n_l;                 // x-lines per tile
    int S;                   // states per x-line
    int ntile[kMaxDims];     // tiles per position
    int tline[kMaxDims];     // V-line step between consecutive tiles of a position
};

// rows (16-byte planes, local V order)  ->  word-SoA planes in tile order.  One thread per row.
template <int D>
__global__ void __launch_bounds__(kBlock) retile_rows_kernel(const unsigned char* __restrict__ src, long long n_pad_src,
                                                             long long s_begin, unsigned* __restrict__ dst,
                                                             long long plane_words, const int* __restrict__ line_off,
                                                             TileGeo geo, long long tile_begin, long long n_rows) {
    const long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n_rows) return;
    const long long per_tile = (long long)geo.n_l * geo.S;
    const long long tile = r / per_tile;
    const int rem = (int)(r - tile * per_tile);
    const int xl = rem / geo.S, x = rem - xl * geo.S;
    long long t = tile_begin + tile, line = 0;
    for (int k = geo.n_pos - 1; k >= 0; --k) {
        const long long q = t / geo.ntile[k];
        line += (t - q * geo.ntile[k]) * (long long)geo.tline[k];
        t = q;
    }
    const long long v = (line + line_off[xl]) * (long long)geo.S + x;
    unsigned w[Row<D>::W];
    load_row<D>(src, n_pad_src, v - s_begin, w);
#pragma unroll
    for (int k = 0; k < Row<D>::W; ++k) dst[(size_t)k * (size_t)plane_words + (size_t)r] = w[k];
}

__global__ void count_mismatch_kernel(const unsigned* a, const unsigned* b, long long n, unsigned long long* out) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const bool bad = i < n && a[i] != b[i];
    const unsigned m = __ballot_sync(0xffffffffu, bad);
    if ((threadIdx.x & 31) == 0 && m) atomicAdd(out, (unsigned long long)__popc(m));
}

// ---------------------------------------------------------------------------
// Batched policy lookup with get_optimal_action semantics (utils/barycentric.py:11-108).  The per-point
// arithmetic (LookupGrid, lookup_point) lives in lookup_src.cuh, shared with the NVRTC-compiled rollout
// kernels (rollout_src.cuh).  One thread per query point.
// ---------------------------------------------------------------------------
#include "lookup_src.cuh"

__global__ void __launch_bounds__(kBlock) lookup_actions_kernel(LookupGrid g, const float* __restrict__ points, long long n,
                                                                const int* __restrict__ policy,
                                                                const float* __restrict__ actions, float* __restrict__ out) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    out[i] = lookup_point(g, g.n_dims, points + i * g.n_dims, policy, actions);
}

// Warm start (pi_prolong_values): V[s] = the source value function `src` (reference order, grid `sg`, taken as uniform)
// interpolated at the node of state s of this rank's slice, with interp_value_point's arithmetic.  One thread per local
// state in storage order; the node is read from the engine's axes (the float32 bits of states_space).  Absorbing states
// (term[k], the per-state flag the table builder turned into PI_ROW_ABSORBING rows) keep the value they hold.  Writes
// both V buffers.
struct AxisPtrs {
    const float* a[kMaxDims];
};

template <int D>
__global__ void __launch_bounds__(kBlock) prolong_values_kernel(GridDesc g, AxisPtrs axes, LookupGrid sg,
                                                                const float* __restrict__ src,
                                                                const unsigned char* __restrict__ term, long long s_begin,
                                                                long long n_local, float* V0, float* V1) {
    const long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n_local || term[k]) return;
    float x[D];
    long long r = s_begin + k;
#pragma unroll
    for (int j = D - 1; j >= 0; --j) {   // storage position j holds logical dimension perm[j]
        const int d = g.perm[j];
        const long long q = r / g.shape[d];
        const float node = axes.a[d][r - q * g.shape[d]];
        r = q;
#pragma unroll
        for (int e = 0; e < D; ++e)      // x stays in registers: no run-time index into it
            if (e == d) x[e] = node;
    }
    const float v = interp_value_point(sg, D, x, src);
    V0[s_begin + k] = v;
    V1[s_begin + k] = v;
}

// Recorded rollout trajectories (rollout_src.cuh) are staged step-major: a rows x n matrix, row r = t * per + k,
// column = episode.  This writes its transpose out[e][r] (the episode-major host layout) through 32 x 32 shared-memory
// tiles, both sides coalesced, and puts NaN where step t = r / per lies beyond the episode (r >= (length[e] + extra) * per).
// Block 32 x 8; grid.y strides over the rows.
__global__ void __launch_bounds__(256) rollout_unstage_kernel(const float* __restrict__ in, float* __restrict__ out,
                                                              long long rows, long long n, int per, int extra,
                                                              const int* __restrict__ length) {
    __shared__ float tile[32][33];
    const long long e0 = (long long)blockIdx.x * 32;
    for (long long r0 = (long long)blockIdx.y * 32; r0 < rows; r0 += (long long)gridDim.y * 32) {
        for (int j = threadIdx.y; j < 32; j += blockDim.y) {
            const long long r = r0 + j, e = e0 + threadIdx.x;
            if (r < rows && e < n) tile[j][threadIdx.x] = in[r * n + e];
        }
        __syncthreads();
        for (int j = threadIdx.y; j < 32; j += blockDim.y) {
            const long long e = e0 + j, r = r0 + threadIdx.x;
            if (r < rows && e < n)
                out[e * rows + r] = r < ((long long)length[e] + extra) * per ? tile[threadIdx.x][j] : __int_as_float(0x7fc00000);
        }
        __syncthreads();
    }
}

}  // namespace pi
