// plane_sweep_src.cuh — CUDA source of the PLANE-STAGED evaluation sweep (JIT, NVRTC, sm_100a).
//
// The same Bellman backup as policy_eval_kernel_4d/_6d of the reference
// (src/cuda_policy_iteration.py:616-649, :1044-1079) + the max|x-y| reduction (:563-571, :987-995),
// but the 2^D values of V a backup needs are read from SHARED MEMORY, not gathered through the L1:
//
//   * the two fastest-stored dimensions (f0 fastest, f1 next) span a "V-plane" of PS_P = n_f0 * n_f1
//     floats that is contiguous and 16-byte aligned in HBM; the other D-2 dimensions enumerate planes;
//   * one CTA walks chunks of consecutive state-planes.  All states of a plane that take the same
//     action land in the same cell of the outer dimensions when the dynamics are translation-invariant
//     in f0/f1 (cart position and velocity: every cart-pole environment), so a state-plane needs only a
//     handful of V-planes: 2^(D-2) corner planes per distinct successor cell;
//   * those V-planes are brought in by TMA bulk copies (cp.async.bulk.shared::cluster.global, one
//     contiguous 4*PS_P-byte copy per plane, completion on an mbarrier) into PS_NS shared-memory slots.
//     WHICH planes go into WHICH slots and WHEN is a per-policy plan computed once per policy by
//     pi::plane_plan_kernel (plane_plan.cuh): slots are reused between consecutive state-planes
//     (measured on K5: 16 plane loads per state-plane instead of 36), loads whose slot is idle are issued
//     one step ahead ("early") and overlap the previous plane's backups;
//   * a backup then reads its corners with LDS at [slot(cell, outer corner) + in-plane offset + immediate]
//     — one shared-memory wavefront per 32 lanes instead of 2.5 L1 wavefronts per gather — and runs the
//     reference's arithmetic unchanged: w_c = ((((f_0 f_1) f_2) ..) f_{D-1}), ev = fma(w_c, V_c, ev) for c
//     ascending, new_V = fma(gamma, ev, reward)  =>  bit-identical V.
//
// A state whose successor cell could not be staged (more distinct cells in a plane than the plan
// holds, no free slot) is flagged by the planner and gathers from global memory like gp_sweep does.
//
// ITEM MODE (PS_PACK == 2): the planner (pi::plane_items_kernel) regroups the P states of a plane into work items of two
// states, one item per thread.  REGULAR PAIRS — storage neighbours staged in the same cell whose in-plane offsets are o
// (even) and o+1 (x-neighbours that take the same action: 78 % of K5's states under a bang-bang policy): the corners of
// the second state along f0 are the first state's shifted by one float, so a pair reads one aligned 64-bit word and one
// float per (outer corner, f1 corner) instead of 2 x 2 floats, and carries the two states in the two halves of
// mul.rn.f32x2 / fma.rn.f32x2 (each half rounds exactly like the scalar instruction: same bits) — half the instructions
// per backup.  The planner places a pair in the lane that matches the bank pair of its offset, so that the 64-bit load
// of a half-warp is ONE shared-memory wavefront whatever rows and cells its pairs come from (slot pitch = 0 mod 32
// floats).  The unpaired states follow two per item and take the one-state path, one after the other; terminal states
// (value kept) ride along with pair items.
//
// The host prepends (dpb200.cu: plane_preamble):
//   PS_D, PS_P, PS_NS, PS_THREADS (consumer threads = PS_P rounded up to a warp), PS_MINB, PS_LV,
//   PS_PACK, PS_N0 (extent of the fastest dimension), ps_cj[2^D] (outer-corner number of corner c), ps_imm[2^D] (in-plane float offset of corner c),
//   gp_off[2^D] (global V offset of corner c, fallback path);
// and then sweep_common_src.cuh: pi::PsParams, pi::PlaneRec and its limits, the chunk schedule, the shared device helpers.

typedef unsigned long long ps_u64;

enum : unsigned { ps_bad_slot = (unsigned)pi::kPlanBadSlot << 4 };   // staged slot offset of a cell that is not resident

#define PS_W (PS_D + 2)
#define PS_N4 (PS_W / 4)
#define PS_N2 ((PS_W % 4) / 2)
#define PS_C (1 << PS_D)
#define PS_NOC (PS_C / 4)
#ifndef PS_LV
#define PS_LV 2
#endif
#define PS_NT (PS_C >> PS_LV)
#define PS_PLANE_BYTES (PS_P * 4)
#ifndef PS_PF_AHEAD
#define PS_PF_AHEAD 0                // steps ahead whose V-planes are prefetched into L2 (0: off; measured on K5: 1, 2, 3, 5
                                     // steps ahead -> 1.39, 1.44, 1.63, 1.45 ms per sweep vs 1.34 without: the extra plan reads
                                     // delay the producer's trigger and the prefetches compete with the copies)
#endif
#ifndef PS_ROW_PF
#define PS_ROW_PF 3                  // steps ahead whose rows the producer prefetches into L2 (0: off)
#endif
#ifndef PS_PITCH
#define PS_PITCH PS_PLANE_BYTES      // bytes between slots (>= PS_PLANE_BYTES, multiple of 16)
#endif
#define PS_SLOTS_BYTES (PS_NS * PS_PITCH)
#define PS_KSTRIDE 20                // words between the slot offsets of two cells: 16 + 4, so that the 128-bit reads of different
                                     // cells by the lanes of a warp fall into different banks
#define PS_CS_WORDS (pi::kPlanMaxCells * PS_KSTRIDE)
#ifndef PS_NOUT
#define PS_NOUT 4                    // output planes in flight (ring): written by the consumers of step it, stored by TMA after it
#endif

// ------------------------------------------------------------------ mbarrier / TMA bulk copy
__device__ __forceinline__ unsigned ps_saddr(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void ps_mbar_init(ps_u64* b, unsigned count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(ps_saddr(b)), "r"(count) : "memory");
}
__device__ __forceinline__ void ps_mbar_expect(ps_u64* b, unsigned bytes) {
    asm volatile("mbarrier.expect_tx.relaxed.cta.shared::cta.b64 [%0], %1;" ::"r"(ps_saddr(b)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void ps_mbar_arrive_expect(ps_u64* b, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(ps_saddr(b)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void ps_mbar_arrive(ps_u64* b) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(ps_saddr(b)) : "memory");
}
__device__ __forceinline__ void ps_mbar_wait(ps_u64* b, unsigned parity) {
    // try_wait suspends the thread until the phase completes or a hardware time limit passes.  (A longer limit through the
    // suspend-time hint was measured slower: 1.34 vs 1.29 ms per K5 sweep — waking late costs more than polling.)
    asm volatile(
        "{\n\t.reg .pred P1;\n\t"
        "PS_WAIT:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n\t"
        "@P1 bra PS_DONE;\n\t"
        "bra PS_WAIT;\n\t"
        "PS_DONE:\n\t}"
        ::"r"(ps_saddr(b)), "r"(parity) : "memory");
}
// L2 prefetch of one V-plane (no shared-memory slot needed: issued steps ahead of the copy that will use it)
__device__ __forceinline__ void ps_bulk_prefetch_l2(const void* src, unsigned bytes) {
    asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(src), "r"(bytes) : "memory");
}
// one contiguous V-plane: global -> shared, completion bytes on the mbarrier
__device__ __forceinline__ void ps_bulk_load(void* dst, const void* src, unsigned bytes, ps_u64* b) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(ps_saddr(dst)), "l"(src), "r"(bytes), "r"(ps_saddr(b)) : "memory");
}

// one contiguous plane of new values: shared -> global (local V buffer or a peer's, over NVLink), bulk async-group completion
__device__ __forceinline__ void ps_bulk_store(void* dst, const void* src, unsigned bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst), "r"(ps_saddr(src)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void ps_bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void ps_bulk_wait_read() { asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory"); }
__device__ __forceinline__ void ps_bulk_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void ps_fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// row of local state s: word 0 = planner code (prow0), words 1..D = fractions, word D+1 = reward
__device__ __forceinline__ void ps_load_row(const pi::PsParams& p, long long s, unsigned (&w)[PS_W]) {
    {
        const uint4 v = pi::ld_stream16(p.prow0 + (size_t)s * 16u);
        w[0] = v.x; w[1] = v.y; w[2] = v.z; w[3] = v.w;
    }
#pragma unroll
    for (int q = 1; q < PS_N4; ++q) {
        const uint4 v = pi::ld_stream16(p.rows + (size_t)q * 16u * (size_t)p.n_pad + (size_t)s * 16u);
        w[4 * q] = v.x; w[4 * q + 1] = v.y; w[4 * q + 2] = v.z; w[4 * q + 3] = v.w;
    }
#if PS_N2
    {
        const uint2 v = pi::ld_stream8(p.rows + (size_t)PS_N4 * 16u * (size_t)p.n_pad + (size_t)s * 8u);
        w[4 * PS_N4] = v.x; w[4 * PS_N4 + 1] = v.y;
    }
#endif
#if PS_W % 2
    w[PS_W - 1] = pi::ld_stream4(p.rows + ((size_t)PS_N4 * 16u + (size_t)PS_N2 * 8u) * (size_t)p.n_pad + (size_t)s * 4u);
#endif
}

// Fallback: the successor cell of this state is not staged -> gather from global memory (gp_sweep's arithmetic).
// Scalars by value: the row must not be forced into local memory by a call.
__device__ __noinline__ float ps_gather_global(const float* __restrict__ Vin, int base, float f0, float f1, float f2, float f3
#if PS_D >= 5
                                               , float f4
#endif
#if PS_D >= 6
                                               , float f5
#endif
) {
    const float* v = Vin + base;
    float ev = 0.0f;
#pragma unroll 1
    for (int c = 0; c < PS_C; ++c) {
        float leaf = (c & 1) ? f0 : 1.0f - f0;
        leaf = leaf * ((c & 2) ? f1 : 1.0f - f1);
        leaf = leaf * ((c & 4) ? f2 : 1.0f - f2);
        leaf = leaf * ((c & 8) ? f3 : 1.0f - f3);
#if PS_D >= 5
        leaf = leaf * ((c & 16) ? f4 : 1.0f - f4);
#endif
#if PS_D >= 6
        leaf = leaf * ((c & 32) ? f5 : 1.0f - f5);
#endif
        int off = 0;
#pragma unroll
        for (int d = 0; d < PS_D; ++d)
            if ((c >> d) & 1) off += gp_off[1 << d];
        ev = fmaf(leaf, __ldg(v + off), ev);
    }
    return ev;
}


#if PS_PACK == 2
// ------------------------------------------------------------------ item mode
#if PS_N0 % 2
#error "item mode needs rows of even length"
#endif
#define PS_NI PS_THREADS                 // item slots per state-plane (two states each; >= PS_P / 2), one per consumer thread
#define PS_NQ ((2 * PS_W + 3) / 4)       // 16-byte quarters per item
#define PS_KIND(c) (((c) >> 27) & 7u)
#define PS_EMPTY (4u << 27)
// item `t` of local state-plane `pl`: state A in words [0, W), state B in words [W, 2W)
__device__ __forceinline__ void ps_load_item(const pi::PsParams& p, long long pl, int t, unsigned (&u)[4 * PS_NQ]) {
    const unsigned char* src = p.prow0 + ((size_t)pl * PS_NQ * PS_NI + (size_t)t) * 16u;
#pragma unroll
    for (int q = 0; q < PS_NQ; ++q) {
        const uint4 v = pi::ld_stream16(src + (size_t)q * PS_NI * 16u);
        u[4 * q] = v.x; u[4 * q + 1] = v.y; u[4 * q + 2] = v.z; u[4 * q + 3] = v.w;
    }
}
// one state from its staged V-planes: the reference's weight products and fma chain (scalar form of the non-item mode)
__device__ __forceinline__ float ps_backup_one(const unsigned* csk, const unsigned char* sbase, const float (&fr)[PS_D]) {
    float pre[PS_NT];
    pre[0] = 1.0f - fr[0];
    pre[1] = fr[0];
#pragma unroll
    for (int d = 1; d < PS_D - PS_LV; ++d) {
        const float f = fr[d], gq = 1.0f - f;
#pragma unroll
        for (int c = PS_NT / 2 - 1; c >= 0; --c) {
            if (c < (1 << d)) {
                const float t = pre[c];
                pre[c + (1 << d)] = t * f;
                pre[c] = t * gq;
            }
        }
    }
    float wt[PS_LV][2];
#pragma unroll
    for (int q = 0; q < PS_LV; ++q) {
        const float l = fr[PS_D - PS_LV + q];
        wt[q][0] = 1.0f - l;
        wt[q][1] = l;
    }
    float ev = 0.0f;
#pragma unroll
    for (int c = 0; c < PS_C; ++c) {
        float leaf = pre[c & (PS_NT - 1)];
#pragma unroll
        for (int q = 0; q < PS_LV; ++q) leaf = leaf * wt[q][(c >> (PS_D - PS_LV + q)) & 1];
        const float* a = reinterpret_cast<const float*>(sbase + csk[ps_cj[c]]);
        ev = fmaf(leaf, a[ps_imm[c]], ev);
    }
    return ev;
}
// a regular pair: state B's corners are state A's shifted by one float along f0, so corner c of B is the float after
// corner c of A; both states ride in the halves of packed multiplies / fmas (per half: the scalar instruction's rounding)
__device__ __forceinline__ ps_u64 ps_backup_pair(const unsigned* csk, const unsigned char* sbase, const float (&fa)[PS_D],
                                                 const float (&fb)[PS_D]) {
    unsigned cso[PS_NOC];
#pragma unroll
    for (int j = 0; j < PS_NOC; j += 4) {
        const uint4 v = *reinterpret_cast<const uint4*>(csk + j);
        cso[j] = v.x; cso[j + 1] = v.y; cso[j + 2] = v.z; cso[j + 3] = v.w;
    }
    ps_u64 pre[PS_NT];
    pre[0] = pi::pk(1.0f - fa[0], 1.0f - fb[0]);
    pre[1] = pi::pk(fa[0], fb[0]);
#pragma unroll
    for (int d = 1; d < PS_D - PS_LV; ++d) {
        const ps_u64 ff = pi::pk(fa[d], fb[d]), gg = pi::pk(1.0f - fa[d], 1.0f - fb[d]);
#pragma unroll
        for (int c = PS_NT / 2 - 1; c >= 0; --c) {
            if (c < (1 << d)) {
                const ps_u64 t = pre[c];
                pre[c + (1 << d)] = pi::mul2(t, ff);
                pre[c] = pi::mul2(t, gg);
            }
        }
    }
    ps_u64 wt[PS_LV][2];
#pragma unroll
    for (int q = 0; q < PS_LV; ++q) {
        const float la = fa[PS_D - PS_LV + q], lb = fb[PS_D - PS_LV + q];
        wt[q][0] = pi::pk(1.0f - la, 1.0f - lb);
        wt[q][1] = pi::pk(la, lb);
    }
    ps_u64 ev = pi::pk(0.0f, 0.0f);
#pragma unroll
    for (int c = 0; c < PS_C; ++c) {
        ps_u64 leaf = pre[c & (PS_NT - 1)];
#pragma unroll
        for (int q = 0; q < PS_LV; ++q) leaf = pi::mul2(leaf, wt[q][(c >> (PS_D - PS_LV + q)) & 1]);
        const float* a = reinterpret_cast<const float*>(sbase + cso[ps_cj[c]]);
        // the compiler loads each float once: 3 per (outer corner, f1 corner)
        // the planner starts pairs at even in-plane offsets only (rows have even length), so the first two floats are one
        // aligned 64-bit load (lanes two floats apart: a 32-bit load would pay a two-way bank conflict)
        const int i0 = ps_imm[c] & ~1;
        const float2 lo = *reinterpret_cast<const float2*>(a + i0);
        const ps_u64 vv = (ps_imm[c] & 1) ? pi::pk(lo.y, a[i0 + 2]) : pi::pk(lo.x, lo.y);
        ev = pi::fma2(leaf, vv, ev);
    }
    return ev;
}
#endif

#define PS_CWARPS (PS_THREADS / 32)     // consumer warps

// Roles: warps 0 .. PS_CWARPS-1 back up the states of the current plane (thread t <-> state t); the last warp is the
// PRODUCER: it issues the TMA bulk loads of the plan and publishes the slot offsets of each step.
// Synchronisation (no CTA-wide barrier in the loop):
//   full[b]  (tx barrier, one arrival by the producer): the V-planes and slot offsets of step `it` (b = it & 1) are in
//            shared memory.  Early loads of step it+1 are issued — and, when that step has no late loads, the barrier
//            is armed — while step `it` is still being computed, so a warp that finishes early runs one step ahead;
//   done[b]  (PS_CWARPS arrivals): every consumer warp has finished step `it`: its slots may be overwritten.
extern "C" __global__ void __launch_bounds__(PS_THREADS + 32, PS_MINB) ps_sweep(const pi::PsParams p)
{
    extern __shared__ __align__(128) unsigned char ps_smem[];
    unsigned* const cs_s = reinterpret_cast<unsigned*>(ps_smem + PS_SLOTS_BYTES);                    // [2][PS_CS_WORDS] slot byte offsets
    ps_u64* const full = reinterpret_cast<ps_u64*>(ps_smem + PS_SLOTS_BYTES + 2 * PS_CS_WORDS * 4);   // [2]
    ps_u64* const done = full + 2;                                                                   // [2]
    float* const out_s = reinterpret_cast<float*>(ps_smem + PS_SLOTS_BYTES + 2 * PS_CS_WORDS * 4 + 32);   // [PS_NOUT][PS_P] new values of a plane
    __shared__ float s_red[(PS_THREADS + 32) / 32];

    const pi::Ctl* __restrict__ ctl = p.ctl;
    if (ctl->done) return;
    const int par = (ctl->base + p.j + ctl->parity0) & 1;
    const float* __restrict__ Vin = par ? p.V1 : p.V0;
    float* __restrict__ Vout = par ? p.V0 : p.V1;

    const int tid = threadIdx.x, lane = tid & 31;
    const bool is_prod = tid >= PS_THREADS;
    const bool has_state = tid < PS_P;

    if (tid == 0) {
        ps_mbar_init(&full[0], 1);
        ps_mbar_init(&full[1], 1);
        ps_mbar_init(&done[0], PS_CWARPS);
        ps_mbar_init(&done[1], PS_CWARPS);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();

    unsigned it = 0;   // steps this CTA has started: step `it` completes phase (it >> 1) & 1 of full[it & 1] and done[it & 1]
    float res = 0.0f;

    if (is_prod) {
        // ------------------------------------------------------------------ producer warp
        // The producer is idle while the consumers compute: it fetches the plan entries of its NEXT trigger into
        // registers before it waits for the consumers, so the TMA copies go out the moment the slots are free.
        // The plan record of a step (header, load list, slot offsets) is fetched into registers TWO steps before it is used,
        // with independent loads (the whole load list, whatever the counts): the producer's trigger after `done` never waits
        // for global memory.  (Fetching a record when it was needed — header first, then the entries it announces — put two
        // dependent DRAM round trips into every step: the sweep took the same 1.31 ms with half the consumer instructions.)
        constexpr int kPerLane = (pi::kPlanMaxLoads + 31) / 32;
        struct Fetched {
            unsigned hdr;               // n_early | n_late << 8 | n_cells << 16 | flags << 24
            unsigned e[kPerLane];       // loads[lane + 32 q]: early loads first, then the late ones
            uint2 cs;                   // slot offsets of (cell lane / 4, outer corners 4 (lane % 4) ..)
        };
        auto fetch_rec = [&](const pi::PlaneRec* r, Fetched& f) {
            f.hdr = *reinterpret_cast<const unsigned*>(r);
#pragma unroll
            for (int q = 0; q < kPerLane; ++q) f.e[q] = lane + 32 * q < pi::kPlanMaxLoads ? r->loads[lane + 32 * q] : 0u;
            f.cs = *reinterpret_cast<const uint2*>(reinterpret_cast<const unsigned short*>(r->cs) + lane * 4);
        };
        // entries [first, first + n) of the record's list: one TMA bulk copy each
        auto copies = [&](const Fetched& f, unsigned first, unsigned n, ps_u64* bar) {
#pragma unroll
            for (int q = 0; q < kPerLane; ++q) {
                const unsigned t = (unsigned)(lane + 32 * q);
                if (t >= first && t < first + n)
                    ps_bulk_load(ps_smem + (size_t)(f.e[q] >> 24) * PS_PITCH, Vin + (size_t)(f.e[q] & 0xffffffu) * PS_P, PS_PLANE_BYTES, bar);
            }
        };
        auto stage_cs_regs = [&](const uint2 v, unsigned buf) {
            uint4 o;
            o.x = (v.x & 0xffffu) << 4; o.y = (v.x >> 16) << 4; o.z = (v.y & 0xffffu) << 4; o.w = (v.y >> 16) << 4;
            *reinterpret_cast<uint4*>(cs_s + buf * PS_CS_WORDS + (lane >> 2) * PS_KSTRIDE + (lane & 3) * 4) = o;
        };
        // The new values of a plane leave through shared memory too: the consumers write them into out_s[it % PS_NOUT], and once
        // every consumer warp is done with the step this warp stores the whole plane with ONE TMA bulk copy into the local V
        // buffer — and with one more per peer that needs the plane (sharded runs: peer buffers over NVLink; the ranges peers
        // need are rounded to whole planes by the host).  No store instruction of the backup threads touches global memory.
        long long prev_g0 = -1;   // first global state of the plane of the previous step
        auto store_plane = [&](unsigned step, long long g0) {
            if (lane == 0) {
                const float* src = out_s + (size_t)(step % PS_NOUT) * PS_P;
                ps_bulk_store(Vout + g0, src, PS_PLANE_BYTES);
                for (int r = 0; r < p.peers.n; ++r)
                    if (g0 >= p.peers.lo[r] && g0 + PS_P <= p.peers.hi[r])
                        ps_bulk_store((par ? p.peers.V0[r] : p.peers.V1[r]) + g0, src, PS_PLANE_BYTES);
                ps_bulk_commit();
                ps_bulk_wait_read<PS_NOUT - 2>();   // the buffer the consumers may write next (step + 2) has been read out
            }
            __syncwarp();
        };
        // The CTA's steps run on across its chunks: the record of the step after next is fetched, and the next step's early
        // loads are issued, also when that step is the first of the next chunk (the planner stitched the chunks for this
        // sequence).  Only the first step of the launch issues all of its loads itself.
        bool armed = false;   // full[it & 1] was already armed one step ahead
        int f_ci = p.sched_begin + blockIdx.x, f_pl = 0, f_end = 0;   // fetch cursor: the step whose record is fetched next
        if (f_ci < p.sched_end) {
            f_pl = pi::plan_chunk_begin(p, pi::plan_chunk_at(p, f_ci));
            f_end = pi::plan_chunk_begin(p, pi::plan_chunk_at(p, f_ci) + 1);
        }
        auto fetch_next = [&](Fetched& f) {
            if (f_ci >= p.sched_end) return;
            fetch_rec(p.plan + f_pl, f);
            if (++f_pl == f_end) {
                f_ci += gridDim.x;
                if (f_ci < p.sched_end) {
                    f_pl = pi::plan_chunk_begin(p, pi::plan_chunk_at(p, f_ci));
                    f_end = pi::plan_chunk_begin(p, pi::plan_chunk_at(p, f_ci) + 1);
                }
            }
        };
        Fetched cur, nxt, nn;
        fetch_next(cur);
        nxt = cur;
        fetch_next(nxt);
        nn = nxt;
        for (int ci = p.sched_begin + blockIdx.x; ci < p.sched_end; ci += gridDim.x) {
            const int chunk = pi::plan_chunk_at(p, ci);
            const int pl0 = pi::plan_chunk_begin(p, chunk);
            const int Lc = pi::plan_chunk_begin(p, chunk + 1) - pl0;
            const bool next_chunk = ci + (int)gridDim.x < p.sched_end;
            for (int i = 0; i < Lc; ++i, ++it) {
                const bool more = i + 1 < Lc || next_chunk;
                const unsigned b = it & 1;
                fetch_next(nn);   // in flight while this warp waits for the consumers
#if PS_ROW_PF > 0
                // The consumers load the rows of a plane one step before they use them — less than a DRAM round trip once a step
                // takes about a microsecond (ncu: 21 % of the warp samples waited for those loads).  One bulk L2 prefetch per plane,
                // PS_ROW_PF steps ahead (into the CTA's next chunk at the end of a chunk), turns them into L2 hits.
                if (lane == 0) {
                    int pf_pl = pl0 + i + PS_ROW_PF;
                    if (i + PS_ROW_PF >= Lc) {
                        pf_pl = -1;
                        if (next_chunk) {
                            const int chn = pi::plan_chunk_at(p, ci + (int)gridDim.x);
                            pf_pl = pi::plan_chunk_begin(p, chn) + (i + PS_ROW_PF - Lc);
                            if (pf_pl >= pi::plan_chunk_begin(p, chn + 1)) pf_pl = -1;
                        }
                    }
                    if (pf_pl >= 0) {
#if PS_PACK == 2
                        ps_bulk_prefetch_l2(p.prow0 + (size_t)pf_pl * PS_NQ * PS_NI * 16u, PS_NQ * PS_NI * 16u);
#else
                        ps_bulk_prefetch_l2(p.prow0 + (size_t)pf_pl * PS_P * 16u, PS_P * 16u);
#pragma unroll
                        for (int q = 1; q < PS_N4; ++q)
                            ps_bulk_prefetch_l2(p.rows + (size_t)q * 16u * (size_t)p.n_pad + (size_t)pf_pl * PS_P * 16u, PS_P * 16u);
#endif
                    }
                }
#endif
#if PS_PF_AHEAD > 0
                // optional (off by default, see PS_PF_AHEAD): pull the planes of a later step into L2 now
                if (i + PS_PF_AHEAD < Lc) {
                    const pi::PlaneRec* rp = p.plan + pl0 + i + PS_PF_AHEAD;
                    const unsigned np = (unsigned)rp->n_early + rp->n_late;
                    for (unsigned q = lane; q < np; q += 32)
                        ps_bulk_prefetch_l2(Vin + (size_t)(rp->loads[q] & 0xffffffu) * PS_P, PS_PLANE_BYTES);
                }
#endif
                const unsigned ne = cur.hdr & 0xffu, nl = (cur.hdr >> 8) & 0xffu;
                const unsigned ne_n = nxt.hdr & 0xffu, nl_n = (nxt.hdr >> 8) & 0xffu;
                // every consumer warp is done with the previous step: its slots (and the other cs buffer) are free
                if (it > 0) ps_mbar_wait(&done[b ^ 1], ((it - 1) >> 1) & 1);
                if (prev_g0 >= 0) store_plane(it - 1, prev_g0);
                prev_g0 = p.s_begin + (long long)(pl0 + i) * PS_P;
                if (!armed) {
                    // the first step of the launch: nothing was issued ahead, its early loads go out now too
                    const unsigned first = it == 0 ? 0u : ne, n = it == 0 ? ne + nl : nl;
                    stage_cs_regs(cur.cs, b);
                    __syncwarp();
                    if (lane == 0) {
                        if (n) ps_mbar_arrive_expect(&full[b], n * (unsigned)PS_PLANE_BYTES);
                        else ps_mbar_arrive(&full[b]);
                    }
                    __syncwarp();
                    copies(cur, first, n, &full[b]);
                }
                armed = false;
                if (more) {
                    stage_cs_regs(nxt.cs, b ^ 1);
                    __syncwarp();
                    if (lane == 0) {
                        if (nl_n == 0) {   // nothing of the next step waits for this one: arm it now, warps may run ahead
                            if (ne_n) ps_mbar_arrive_expect(&full[b ^ 1], ne_n * (unsigned)PS_PLANE_BYTES);
                            else ps_mbar_arrive(&full[b ^ 1]);
                        } else if (ne_n) {
                            ps_mbar_expect(&full[b ^ 1], ne_n * (unsigned)PS_PLANE_BYTES);
                        }
                    }
                    __syncwarp();
                    copies(nxt, 0u, ne_n, &full[b ^ 1]);
                    armed = nl_n == 0;
                }
                cur = nxt;
                nxt = nn;
            }
        }
        if (prev_g0 >= 0) {   // the last plane of this CTA
            ps_mbar_wait(&done[(it - 1) & 1], ((it - 1) >> 1) & 1);
            store_plane(it - 1, prev_g0);
        }
        if (lane == 0) ps_bulk_wait_all();   // every plane of new values has landed before the kernel ends
    } else {
        // ------------------------------------------------------------------ consumer warps
#if PS_PACK == 2
        // the item of the CTA's next step is in flight while this one is backed up, across chunk boundaries too
        unsigned u[4 * PS_NQ];
        if (p.sched_begin + (int)blockIdx.x < p.sched_end)
            ps_load_item(p, pi::plan_chunk_begin(p, pi::plan_chunk_at(p, p.sched_begin + blockIdx.x)), tid, u);
        for (int ci = p.sched_begin + blockIdx.x; ci < p.sched_end; ci += gridDim.x) {
            const int chunk = pi::plan_chunk_at(p, ci);
            const int pl0 = pi::plan_chunk_begin(p, chunk);
            const int Lc = pi::plan_chunk_begin(p, chunk + 1) - pl0;
            const int pl_next = ci + (int)gridDim.x < p.sched_end ? pi::plan_chunk_begin(p, pi::plan_chunk_at(p, ci + (int)gridDim.x)) : -1;
            for (int i = 0; i < Lc; ++i, ++it) {
                const unsigned b = it & 1;
                const long long sp = (long long)(pl0 + i) * PS_P;   // first local state of the plane
                const long long g0 = p.s_begin + sp;
                const unsigned c0 = u[0];
                const bool is_pair = (c0 >> 31) != 0u;
                // An item on the pair path: the second state has the next in-plane index and the next offset in the same cell;
                // bits 27-28 say which halves hold a state (0 both, 1 the first only, 2 the second only — a single with a
                // dummy partner whose result is dropped); the second code word carries a passenger (a terminal state, whose
                // value is kept) or nothing.
                const unsigned vm = (c0 >> 27) & 3u;
                const unsigned ca = is_pair ? (c0 & 0x87ffffffu) | (vm == 2u ? PS_EMPTY : 0u) : c0;
                const unsigned cb = is_pair ? ((c0 & 0x07ffffffu) + 0x1001u) | (vm == 1u ? PS_EMPTY : 0u) : u[PS_W];
                const unsigned pass = is_pair ? u[PS_W] : 0u;
                float fa[PS_D], fb[PS_D];
#pragma unroll
                for (int d = 0; d < PS_D; ++d) { fa[d] = __uint_as_float(u[1 + d]); fb[d] = __uint_as_float(u[PS_W + 1 + d]); }
                const float ra = __uint_as_float(u[PS_D + 1]), rb = __uint_as_float(u[PS_W + PS_D + 1]);
                // the next plane's item: in flight while this one is backed up
                if (i + 1 < Lc) ps_load_item(p, pl0 + i + 1, tid, u);
                else if (pl_next >= 0) ps_load_item(p, pl_next, tid, u);
                const unsigned kinda = PS_KIND(ca), kindb = PS_KIND(cb);
                const unsigned pa = ca & 0xfffu, pb = cb & 0xfffu;
                float volda = 0.0f, voldb = 0.0f, vpass = 0.0f;
                if (kinda < 4u && (p.check || kinda == 3u)) volda = Vin[g0 + pa];
                if (kindb < 4u && (p.check || kindb == 3u)) voldb = Vin[g0 + pb];
                if (pass >> 31) vpass = Vin[g0 + (pass & 0xfffu)];

                ps_mbar_wait(&full[b], (it >> 1) & 1);

                float eva = 0.0f, evb = 0.0f;
                const unsigned* csa = cs_s + b * PS_CS_WORDS + ((ca >> 24) & 7u) * PS_KSTRIDE;
                if (is_pair && csa[0] != ps_bad_slot) {
                    const ps_u64 ev2 = ps_backup_pair(csa, ps_smem + ((ca >> 12) & 0xfffu) * 4u, fa, fb);
                    pi::unpk(ev2, eva, evb);
                } else {
#pragma unroll 1
                    for (int h = 0; h < 2; ++h) {
                        const unsigned cc = h ? cb : ca;
                        const unsigned kind = PS_KIND(cc);
                        if (kind > 1u) continue;   // terminated (sum = 0), terminal (V kept) or no state
                        float fr[PS_D];
#pragma unroll
                        for (int d = 0; d < PS_D; ++d) fr[d] = h ? fb[d] : fa[d];
                        const unsigned* csk = cs_s + b * PS_CS_WORDS + ((cc >> 24) & 7u) * PS_KSTRIDE;
                        float ev;
                        if (kind == 0u && csk[0] != ps_bad_slot) {
                            ev = ps_backup_one(csk, ps_smem + ((cc >> 12) & 0xfffu) * 4u, fr);
                        } else {
                            // not staged: the original base index is word 0 of the policy's row
                            const int base = (int)pi::ld_stream4(p.rows + (size_t)(sp + (cc & 0xfffu)) * 16u);
                            ev = ps_gather_global(Vin, base, fr[0], fr[1], fr[2], fr[3]
#if PS_D >= 5
                                                  , fr[4]
#endif
#if PS_D >= 6
                                                  , fr[5]
#endif
                            );
                        }
                        if (h) evb = ev; else eva = ev;
                    }
                }
                float* const o = out_s + (it % PS_NOUT) * PS_P;
                if (kinda < 4u) {
                    const float vnew = kinda == 3u ? volda : fmaf(p.gamma, eva, ra);
                    o[pa] = vnew;
                    if (p.check) res = fmaxf(res, fabsf(vnew - volda));
                }
                if (kindb < 4u) {
                    const float vnew = kindb == 3u ? voldb : fmaf(p.gamma, evb, rb);
                    o[pb] = vnew;
                    if (p.check) res = fmaxf(res, fabsf(vnew - voldb));
                }
                if (pass >> 31) o[pass & 0xfffu] = vpass;
                ps_fence_async_smem();   // the plane is read by the TMA store (async proxy)
                __syncwarp();
                if (lane == 0) ps_mbar_arrive(&done[b]);
            }
        }
#else
        // the row of the CTA's next step is in flight while this one is backed up, across chunk boundaries too
        unsigned w[PS_W];
        if (has_state && p.sched_begin + (int)blockIdx.x < p.sched_end)
            ps_load_row(p, (long long)pi::plan_chunk_begin(p, pi::plan_chunk_at(p, p.sched_begin + blockIdx.x)) * PS_P + tid, w);
        for (int ci = p.sched_begin + blockIdx.x; ci < p.sched_end; ci += gridDim.x) {
            const int chunk = pi::plan_chunk_at(p, ci);
            const int pl0 = pi::plan_chunk_begin(p, chunk);
            const int Lc = pi::plan_chunk_begin(p, chunk + 1) - pl0;
            const int pl_next = ci + (int)gridDim.x < p.sched_end ? pi::plan_chunk_begin(p, pi::plan_chunk_at(p, ci + (int)gridDim.x)) : -1;
            for (int i = 0; i < Lc; ++i, ++it) {
                const unsigned b = it & 1;
                const long long s = (long long)(pl0 + i) * PS_P + tid;   // local state
                const long long g = p.s_begin + s;
                const int code = has_state ? (int)w[0] : -1;
                const bool staged = code >= 0 && !(code & pi::kPlanFallback);
                const unsigned k = staged ? ((unsigned)code >> 16) : 0u;
                const unsigned ip = staged ? ((unsigned)code & 0xffffu) : 0u;
                float fr[PS_D];
#pragma unroll
                for (int d = 0; d < PS_D; ++d) fr[d] = __uint_as_float(w[1 + d]);
                const float reward = __uint_as_float(w[PS_D + 1]);
                // the next plane's row: in flight while this plane is backed up
                if (i + 1 < Lc && has_state) ps_load_row(p, s + PS_P, w);
                else if (pl_next >= 0 && has_state) ps_load_row(p, (long long)pl_next * PS_P + tid, w);
                float vold = 0.0f;
                if (has_state && (p.check || code == -2)) vold = Vin[g];

                ps_mbar_wait(&full[b], (it >> 1) & 1);

                float ev = 0.0f;
                // a cell whose V-planes found no slot is marked in its slot offsets (plane_slots_kernel): gather from global
                const bool resident = staged && cs_s[b * PS_CS_WORDS + k * PS_KSTRIDE] != ps_bad_slot;
                if (resident) {
                    const unsigned* csk = cs_s + b * PS_CS_WORDS + k * PS_KSTRIDE;
                    const unsigned char* sbase = ps_smem + ip * 4u;
#if PS_PACK
                    // weight tree in packed pairs (corner bit 0 = the two halves): level d multiplies every pair by
                    // (1-f_d, 1-f_d) and (f_d, f_d) — one mul.rn.f32x2 per two products, each half rounded like the
                    // scalar product of the reference
                    ps_u64 node[PS_NT / 2];
                    node[0] = pi::pk(1.0f - fr[0], fr[0]);
#pragma unroll
                    for (int d = 1; d < PS_D - PS_LV; ++d) {
                        const ps_u64 ff = pi::pk(fr[d], fr[d]), gg = pi::pk(1.0f - fr[d], 1.0f - fr[d]);
#pragma unroll
                        for (int c = PS_NT / 4 - 1; c >= 0; --c) {
                            if (c < (1 << (d - 1))) {
                                const ps_u64 t = node[c];
                                node[c + (1 << (d - 1))] = pi::mul2(t, ff);
                                node[c] = pi::mul2(t, gg);
                            }
                        }
                    }
                    ps_u64 wt[PS_LV][2];
#pragma unroll
                    for (int q = 0; q < PS_LV; ++q) {
                        const float l = fr[PS_D - PS_LV + q];
                        wt[q][0] = pi::pk(1.0f - l, 1.0f - l);
                        wt[q][1] = pi::pk(l, l);
                    }
#pragma unroll
                    for (int c = 0; c < PS_C; c += 2) {
                        ps_u64 leaf = node[(c & (PS_NT - 1)) >> 1];
#pragma unroll
                        for (int q = 0; q < PS_LV; ++q) leaf = pi::mul2(leaf, wt[q][(c >> (PS_D - PS_LV + q)) & 1]);
                        float l0, l1;
                        pi::unpk(leaf, l0, l1);
                        const float* a0 = reinterpret_cast<const float*>(sbase + csk[ps_cj[c]]);
                        const float* a1 = reinterpret_cast<const float*>(sbase + csk[ps_cj[c + 1]]);
                        ev = fmaf(l0, a0[ps_imm[c]], ev);
                        ev = fmaf(l1, a1[ps_imm[c + 1]], ev);
                    }
#else
                    float pre[PS_NT];
                    pre[0] = 1.0f - fr[0];
                    pre[1] = fr[0];
#pragma unroll
                    for (int d = 1; d < PS_D - PS_LV; ++d) {
                        const float f = fr[d], gq = 1.0f - f;
#pragma unroll
                        for (int c = PS_NT / 2 - 1; c >= 0; --c) {
                            if (c < (1 << d)) {
                                const float t = pre[c];
                                pre[c + (1 << d)] = t * f;
                                pre[c] = t * gq;
                            }
                        }
                    }
                    float wt[PS_LV][2];
#pragma unroll
                    for (int q = 0; q < PS_LV; ++q) {
                        const float l = fr[PS_D - PS_LV + q];
                        wt[q][0] = 1.0f - l;
                        wt[q][1] = l;
                    }
#pragma unroll
                    for (int c = 0; c < PS_C; ++c) {
                        float leaf = pre[c & (PS_NT - 1)];
#pragma unroll
                        for (int q = 0; q < PS_LV; ++q) leaf = leaf * wt[q][(c >> (PS_D - PS_LV + q)) & 1];
                        const float* a = reinterpret_cast<const float*>(sbase + csk[ps_cj[c]]);
                        ev = fmaf(leaf, a[ps_imm[c]], ev);
                    }
#endif
                } else if (code >= 0) {
                    // not staged: the original base index is word 0 of the policy's row
                    const int base = (int)pi::ld_stream4(p.rows + (size_t)s * 16u);
                    ev = ps_gather_global(Vin, base, fr[0], fr[1], fr[2], fr[3]
#if PS_D >= 5
                                          , fr[4]
#endif
#if PS_D >= 6
                                          , fr[5]
#endif
                    );
                }
                if (has_state) {
                    const float vnew = code == -2 ? vold : fmaf(p.gamma, ev, reward);
                    out_s[(it % PS_NOUT) * PS_P + tid] = vnew;
                    if (p.check) res = fmaxf(res, fabsf(vnew - vold));
                }
                ps_fence_async_smem();   // the plane is read by the TMA store (async proxy)
                __syncwarp();
                if (lane == 0) ps_mbar_arrive(&done[b]);
            }
        }
#endif
    }

    if (!p.check) return;
    res = pi::warp_max(res);
    if (lane == 0) s_red[tid >> 5] = res;
    __syncthreads();
    if (tid < 32) {
        float r = tid < (PS_THREADS + 32) / 32 ? s_red[tid] : 0.0f;
        r = pi::warp_max(r);
        if (tid == 0) p.partial[p.partial_off + blockIdx.x] = r;
    }
}
