// plane_plan.cuh — per-policy plan of the plane-staged evaluation sweep (plane_sweep_src.cuh).
//
// The policy's rows are fixed for the thousands of sweeps of one policy evaluation
// (src/cuda_policy_iteration.py:300-336), so everything the sweep needs to know about WHICH V-planes
// a state-plane reads is computed once per policy, here, instead of once per sweep:
//
//   * for every state-plane (the PS_P states that share their outer-dimension indices) the distinct
//     successor cells of the outer dimensions (<= kPlanMaxCells) and, per state, the code word
//     (cell number << 16 | in-plane offset of the lower corner) that replaces the row's base index;
//   * a shared-memory slot for each of the 2^(D-2) corner V-planes of every cell, assigned while
//     walking the chunk's state-planes in order: a V-plane already resident from the previous
//     state-plane keeps its slot (no load), a new one takes an idle slot — "early" when the slot was
//     not read by the previous state-plane either (the load overlaps that plane's backups), "late"
//     when it only becomes free once the previous plane is done;
//   * cells that do not fit (more than kPlanMaxCells per plane, no slot left) are flagged: their states
//     gather from global memory in the sweep.
//
// Two passes: plane_cells_kernel (one CTA per state-plane, fully parallel, memory-bound) finds the cells and writes
// the code words; plane_slots_kernel (one warp per chunk of consecutive state-planes, sequential over the chunk
// because the slot state of step i depends on step i-1) assigns slots and writes the load lists.  Every chunk is planned
// as if it started cold; plane_stitch_kernel and plane_relabel_kernel then renumber the slots of each chunk so that the
// first step's loads go to slots the CTA's previous chunk no longer reads, and issue those loads one step ahead too.
#pragma once

#include <cuda_runtime.h>

#include "sweep_common_src.cuh"   // PlaneRec, its limits and the chunk schedule (plan_chunk_begin)

namespace pi {

constexpr int kPlanMaxSlots = 80;
constexpr int kPlanHash = 32;
constexpr int kPlanThreads = 256;

// Per state-plane: its distinct successor cells (lower-corner V-plane numbers) and how many states fall into each.
struct PlaneCells {
    int n_cells;                             // <= kPlanMaxCells
    int n_unstaged;                          // live states whose cell did not fit (more than kPlanMaxCells distinct cells)
    int vp[kPlanMaxCells];
    unsigned short cnt[kPlanMaxCells];
    int pad[2];
};
static_assert(sizeof(PlaneCells) == 64, "PlaneCells layout");

// Per chunk: the slots its first step loads and the slots its last step reads (bit s of 128 = slot s), written by
// plane_slots_kernel; and the renumbering plane_stitch_kernel chose for it.
struct ChunkSlots {
    unsigned first[4];
    unsigned last[4];
};
struct ChunkStitch {
    unsigned busy[4];                        // slots (new numbers) the previous chunk of the same CTA reads in its last step
    unsigned char perm[kPlanMaxSlots];       // planned slot -> slot
    int relabel;                             // 0: the CTA's first chunk, kept as planned
    int pad[3];
};

struct PlanParams {
    const unsigned char* rows;   // the policy's rows; plane 0 = [base, f0, f1, f2] per state (16 B)
    unsigned char* prow0;        // out: [code, f0, f1, f2]
    PlaneRec* plan;              // out: one record per local state-plane
    PlaneCells* cells;           // scratch: one per local state-plane (written by plane_cells_kernel)
    unsigned long long* stats;   // out (atomic): [0] plane loads, [1] late loads, [2] fallback states, [3] live states,
                                 //               [4] staged cells, [5] state-planes
    ChunkSlots* chunk_slots;     // out: one per chunk
    ChunkStitch* stitch;         // one per chunk (plane_stitch_kernel -> plane_relabel_kernel)
    int n_planes;                // local state-planes
    int pl_begin;                // this launch plans the state-planes [pl_begin, pl_end) = the chunks [c_begin, c_end): a policy
    int pl_end;                  // upload is planned range by range while the rest is still on its way (pi_upload_policy_local)
    int c_begin, c_end;
    int L, n_full, n_chunks;     // chunk geometry (plan_chunk_begin)
    int grid, chunk_rot;         // the sweep's schedule: CTA b takes the chunks (b + chunk_rot), (b + G + chunk_rot), ... mod n_chunks
    int P;                       // states per plane
    int NS;                      // shared-memory slots of the sweep
    int noc;                     // outer corners per cell (power of two)
    int pitch;                   // floats between slots in shared memory (>= P, multiple of 4)
    int ooff[kPlanMaxOC];        // V-plane offset of outer corner j
    // item mode (plane_items_kernel): the states of a plane regrouped into P/2 work items of two states each
    unsigned char* irows;        // out: [plane][quarter q < nq][item slot < T] of 16 bytes
    long long n_pad;             // states per row plane of `rows`
    int W;                       // words per row (D + 2)
    int nq;                      // 16-byte quarters per item: ceil(2 W / 4)
    int T;                       // item slots per state-plane = consumer threads of the sweep (>= P / 2, <= 512)
    int hcap;                    // half-warps that may take bank-aligned items (T / 16; the kernel keeps the last ones free for generic items)
};

// Pass 1 — fully parallel, one CTA per state-plane: the distinct successor cells of the plane and the code word of every
// state (cell number << 16 | in-plane offset of the lower corner).  Memory-bound: reads and rewrites the first row plane.
constexpr int kCellThreads = 128;
__global__ void __launch_bounds__(kCellThreads) plane_cells_kernel(const PlanParams q) {
    __shared__ int htab[kPlanHash];             // distinct successor cells of the plane (open addressing)
    __shared__ int hcnt[kPlanHash];
    __shared__ int hcell[kPlanHash];            // hash entry -> cell number (or -1: does not fit)
    const int tid = threadIdx.x, lane = tid & 31;
    const int pl = q.pl_begin + blockIdx.x;
    const long long s0 = (long long)pl * q.P;
    if (tid < kPlanHash) { htab[tid] = -1; hcnt[tid] = 0; hcell[tid] = -1; }
    __syncthreads();
    constexpr int kPer = 8;   // states per thread (P <= 1024)
    uint4 w[kPer];
    int hs[kPer];
#pragma unroll
    for (int r = 0; r < kPer; ++r) {
        const int t = tid + r * kCellThreads;
        hs[r] = -1;
        w[r] = make_uint4(0xfffffffeu, 0u, 0u, 0u);
        if (t < q.P) w[r] = *reinterpret_cast<const uint4*>(q.rows + (size_t)(s0 + t) * 16u);
    }
#pragma unroll
    for (int r = 0; r < kPer; ++r) {
        const int t = tid + r * kCellThreads;
        const int base = (int)w[r].x;
        const bool live = t < q.P && base >= 0;
        const int vp = live ? base / q.P : -1;
        // one insertion per distinct cell per warp: the lanes of a warp mostly share 1-3 cells
        const unsigned act = __ballot_sync(0xffffffffu, live);
        if (live) {
            const unsigned same = __match_any_sync(act, vp);
            int h = -1;
            if ((__ffs(same) - 1) == lane) {
                h = (int)(((unsigned)vp * 2654435761u) >> 27);
                bool ok = false;
                for (int probe = 0; probe < kPlanHash && !ok; ++probe) {
                    const int old = atomicCAS(&htab[h], -1, vp);
                    ok = old == -1 || old == vp;
                    if (!ok) h = (h + 1) & (kPlanHash - 1);
                }
                if (ok) atomicAdd(&hcnt[h], __popc(same));
                else h = -1;
            }
            hs[r] = __shfl_sync(same, h, __ffs(same) - 1);
        }
    }
    __syncthreads();
    if (tid < 32) {   // number the occupied entries; the first kPlanMaxCells become the plane's cells
        const bool occ = htab[lane] != -1;
        const unsigned m = __ballot_sync(0xffffffffu, occ);
        const int k = __popc(m & ((1u << lane) - 1u));
        PlaneCells* pc = q.cells + pl;
        if (occ && k < kPlanMaxCells) {
            hcell[lane] = k;
            pc->vp[k] = htab[lane];
            pc->cnt[k] = (unsigned short)min(hcnt[lane], 65535);
        }
        const int K = min(__popc(m), kPlanMaxCells);
        if (lane >= K && lane < kPlanMaxCells) { pc->vp[lane] = -1; pc->cnt[lane] = 0; }
        if (lane == 0) pc->n_cells = K;
    }
    __syncthreads();
    int n_unstaged = 0;
#pragma unroll
    for (int r = 0; r < kPer; ++r) {
        const int t = tid + r * kCellThreads;
        if (t < q.P) {
            int code = (int)w[r].x;
            if (code >= 0) {
                const int k = hs[r] >= 0 ? hcell[hs[r]] : -1;
                if (k >= 0) code = (k << 16) | (code - (code / q.P) * q.P);
                else { code = kPlanFallback; ++n_unstaged; }
            }
            *reinterpret_cast<uint4*>(q.prow0 + (size_t)(s0 + t) * 16u) = make_uint4((unsigned)code, w[r].y, w[r].z, w[r].w);
        }
    }
    // states outside every cell (rare: more than kPlanMaxCells distinct cells in a plane)
    const unsigned any = __ballot_sync(0xffffffffu, n_unstaged > 0);
    __shared__ int s_un;
    if (tid == 0) s_un = 0;
    __syncthreads();
    if (any && n_unstaged) atomicAdd(&s_un, n_unstaged);
    __syncthreads();
    if (tid == 0) q.cells[pl].n_unstaged = s_un;
}

// Pass 1, ITEM MODE (PS_PACK == 2 in plane_sweep_src.cuh) — one CTA per state-plane.  Besides the cells it regroups the
// plane's P states into work items of two states, one item per sweep thread (T item slots per plane, T >= P / 2):
//   * REGULAR PAIRS: states p and p+1 that are staged in the same successor cell with in-plane offsets o (even) and o+1
//     (x-neighbours that take the same action).  The sweep backs both up from one aligned 64-bit load + one 32-bit load
//     per (outer corner, f1 corner) instead of 2 x 2 loads, with the two states in the halves of packed f32x2 multiplies
//     and fmas.  BANK-ALIGNED PLACEMENT: the 64-bit load of the 16 lanes of a half-warp is one shared-memory wavefront
//     only if the lanes hit 16 distinct bank pairs, so a pair goes to lane (o / 2) mod 16 of the first half-warp in which
//     that lane is free (slot pitch = 0 mod 32 floats: the bank does not depend on the slot, cells may mix in a warp).
//     Natural order pays 2 wavefronts per load (a row of 18 live states is 9 pairs: every half-warp straddles a row break);
//     aligned placement 1.27 at 78 % lane occupancy (scripts/analysis/pair_pack_model.py).  An item that finds its lane
//     taken in every half-warp ("stray": 5 of 205 per K5 plane) takes a free lane of the last, emptiest half-warps —
//     correct anywhere, it only risks a bank conflict with the rightful owner of its class;
//   * STAGED SINGLES (no partner: the neighbour takes another action, or the offset is odd) take the same path with a DUMMY
//     partner — (single, dummy) at an even offset, (dummy, single) one offset back at an odd one — and are placed like
//     pairs, as many as the T slots allow (a single then costs a whole slot instead of half of one);
//   * the LEFTOVER states (global-gather fallback, terminated rows, singles and terminal states that found no seat), two
//     per generic item, fill the free slots from the END: those that need a backup first, the trivial ones last, item j
//     taking leftover j and leftover m-1-j; the sweep runs its one-state path twice for such an item;
//   * TERMINAL states (V kept) ride along as PASSENGERS of pair items (the second state's code word is redundant in a pair).
// Every state keeps its own row words (fractions, reward): nothing about the arithmetic changes, only which thread does
// it.  The code word of a state: bits 0-11 in-plane index p, 12-23 in-plane offset o of the successor's lower corner,
// 24-26 cell number, 27-29 kind (0 staged, 1 global gather, 2 terminated: sum = 0, 3 terminal: V kept, 4 no state),
// bit 31 (first state of an item only): the item takes the pair path — bits 27-28 then say which halves hold a state
// (0 both, 1 the first only, 2 the second only: a single with a dummy partner), the second state's code is the first's
// plus one index and one offset, and the second code word is 0x80000000 | p of the passenger, or kItemEmpty.
constexpr unsigned kItemKindShift = 27;
constexpr unsigned kItemEmpty = 4u << kItemKindShift;
constexpr unsigned kItemPair = 0x80000000u;
constexpr int kItemThreads = 128;
constexpr int kItemSlotsPer = 4;  // item slots per thread (T <= 512)

__device__ __forceinline__ unsigned long long block_excl_scan_u64(unsigned long long v, unsigned long long* s_w, unsigned long long* total) {
    // exclusive sum over the kItemThreads threads of the CTA (s_w: kItemThreads / 32 words of shared memory)
    const int lane = threadIdx.x & 31, wq = threadIdx.x >> 5;
    unsigned long long inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const unsigned long long t = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += t;
    }
    __syncthreads();   // s_w may still be read from a previous scan
    if (lane == 31) s_w[wq] = inc;
    __syncthreads();
    unsigned long long before = 0, all = 0;
#pragma unroll
    for (int w = 0; w < kItemThreads / 32; ++w) {
        const unsigned long long t = s_w[w];
        if (w < wq) before += t;
        all += t;
    }
    *total = all;
    return before + inc - v;
}

// KP = states per thread (the smallest power of two with KP * kItemThreads >= P)
template <int KP>
__global__ void __launch_bounds__(kItemThreads, 8) plane_items_kernel(const PlanParams q) {
    extern __shared__ __align__(16) unsigned char it_smem[];
    __shared__ int htab[kPlanHash];
    __shared__ int hcnt[kPlanHash];
    __shared__ int hcell[kPlanHash];
    __shared__ unsigned long long s_scan[kItemThreads / 32];
    __shared__ int s_un;
    const int P = q.P, T = q.T, W = q.W;
    unsigned* const stage = reinterpret_cast<unsigned*>(it_smem);                                    // [nq][T][4] words
    unsigned* const s_code = stage + (size_t)q.nq * T * 4;                                            // [P]
    unsigned short* const s_dst = reinterpret_cast<unsigned short*>(s_code + P);                     // [P] item slot * 2 + half
    unsigned short* const s_hslot = s_dst + P;                                                        // [P / 2] pair number -> item slot
    unsigned short* const s_free = s_hslot + P / 2;                                                   // [T] free item slots, ascending
    unsigned char* const s_flag = reinterpret_cast<unsigned char*>(s_free + T);                      // [P]
    unsigned char* const s_occ = s_flag + P;                                                          // [T]
    const int tid = threadIdx.x, lane = tid & 31;
    const int pl = q.pl_begin + blockIdx.x;
    const long long s0 = (long long)pl * P;
    if (tid < kPlanHash) { htab[tid] = -1; hcnt[tid] = 0; hcell[tid] = -1; }
    if (tid == 0) s_un = 0;
    __syncthreads();

    // ---- A. the distinct successor cells (as plane_cells_kernel) -> code word of every state
    int w0[KP];   // base word of the row (the other words are read again in phase D: registers matter more than L2 hits)
    int hs[KP];
#pragma unroll
    for (int r = 0; r < KP; ++r) {
        const int t = tid + r * kItemThreads;
        hs[r] = -1;
        w0[r] = -2;
        if (t < P) w0[r] = *reinterpret_cast<const int*>(q.rows + (size_t)(s0 + t) * 16u);
    }
#pragma unroll
    for (int r = 0; r < KP; ++r) {
        const int t = tid + r * kItemThreads;
        const int base = w0[r];
        const bool live = t < P && base >= 0;
        const int vp = live ? base / P : -1;
        const unsigned act = __ballot_sync(0xffffffffu, live);
        if (live) {
            const unsigned same = __match_any_sync(act, vp);
            int h = -1;
            if ((__ffs(same) - 1) == lane) {
                h = (int)(((unsigned)vp * 2654435761u) >> 27);
                bool ok = false;
                for (int probe = 0; probe < kPlanHash && !ok; ++probe) {
                    const int old = atomicCAS(&htab[h], -1, vp);
                    ok = old == -1 || old == vp;
                    if (!ok) h = (h + 1) & (kPlanHash - 1);
                }
                if (ok) atomicAdd(&hcnt[h], __popc(same));
                else h = -1;
            }
            hs[r] = __shfl_sync(same, h, __ffs(same) - 1);
        }
    }
    __syncthreads();
    if (tid < 32) {
        const bool occ = htab[lane] != -1;
        const unsigned m = __ballot_sync(0xffffffffu, occ);
        const int k = __popc(m & ((1u << lane) - 1u));
        PlaneCells* pc = q.cells + pl;
        if (occ && k < kPlanMaxCells) {
            hcell[lane] = k;
            pc->vp[k] = htab[lane];
            pc->cnt[k] = (unsigned short)min(hcnt[lane], 65535);
        }
        const int K = min(__popc(m), kPlanMaxCells);
        if (lane >= K && lane < kPlanMaxCells) { pc->vp[lane] = -1; pc->cnt[lane] = 0; }
        if (lane == 0) pc->n_cells = K;
    }
    __syncthreads();
    int n_unstaged = 0;
#pragma unroll
    for (int r = 0; r < KP; ++r) {
        const int t = tid + r * kItemThreads;
        if (t < P) {
            const int base = w0[r];
            unsigned code = (unsigned)t;
            if (base >= 0) {
                const int k = hs[r] >= 0 ? hcell[hs[r]] : -1;
                if (k >= 0) code |= ((unsigned)(base - (base / P) * P) << 12) | ((unsigned)k << 24);
                else { code |= 1u << kItemKindShift; ++n_unstaged; }
            } else {
                code |= (base == -1 ? 2u : 3u) << kItemKindShift;
            }
            s_code[t] = code;
        }
    }
    if (n_unstaged) atomicAdd(&s_un, n_unstaged);
    // every item slot starts empty: no state in either half, no passenger
    for (int i = tid; i < T; i += kItemThreads) {
        stage[(size_t)i * 4] = kItemEmpty;                                       // word 0 of the item: first state's code
        stage[((size_t)(W >> 2) * T + i) * 4 + (W & 3)] = kItemEmpty;            // word W: second state's code
        s_occ[i] = 0;
    }
    __syncthreads();

    // ---- B. regular pairs (thread <-> KP consecutive states from here on).  A pair starts at an EVEN in-plane
    // offset; offsets grow by one from a state to its partner, so no state is claimed twice
    const int p0 = tid * KP;
    unsigned codes[KP + 1];
#pragma unroll
    for (int i = 0; i <= KP; ++i) codes[i] = p0 + i < P ? s_code[p0 + i] : kItemEmpty;
    unsigned heads = 0;
#pragma unroll
    for (int i = 0; i < KP; ++i) {
        const unsigned a = codes[i], b = codes[i + 1];
        const bool l = (a >> kItemKindShift) == 0u && (b >> kItemKindShift) == 0u && ((a ^ b) & (7u << 24)) == 0u &&
                       ((b >> 12) & 0xfffu) == ((a >> 12) & 0xfffu) + 1u;
        if (l && ((a >> 12) & 1u) == 0u) heads |= 1u << i;
    }
#pragma unroll
    for (int i = 0; i < KP; ++i)
        if (p0 + i < P) s_flag[p0 + i] = (unsigned char)((heads >> i) & 1u);
    __syncthreads();
    unsigned tails = 0;
#pragma unroll
    for (int i = 0; i < KP; ++i) {
        const int p = p0 + i;
        if (p > 0 && p < P && s_flag[p - 1]) tails |= 1u << i;
    }
    __syncthreads();   // s_flag is rewritten below

    // ---- C. item slots.  Round 1 (one exclusive scan over the states in storage order, 12-bit counters): pairs, staged
    // singles, other states that need a backup (global-gather fallback), terminated states, terminal states
    enum { kHead = 0, kTail = 1, kSingle = 2, kWork = 3, kK2 = 4, kK3 = 5 };
    int cat[KP];
    unsigned long long c0 = 0;
#pragma unroll
    for (int i = 0; i < KP; ++i) {
        cat[i] = -1;
        if (p0 + i >= P) continue;
        const unsigned kind = (codes[i] >> kItemKindShift) & 7u;
        // a staged single can ride the pair path (below) unless the dummy in front of it would be state -1
        const bool odd_at_0 = p0 + i == 0 && ((codes[i] >> 12) & 1u);
        cat[i] = ((heads >> i) & 1u) ? kHead : ((tails >> i) & 1u) ? kTail : (kind == 0u && !odd_at_0) ? kSingle : kind <= 1u ? kWork : kind == 2u ? kK2 : kK3;
        if (cat[i] != kTail) c0 += 1ull << (12 * (cat[i] == kHead ? 0 : cat[i] - 1));
    }
    unsigned long long t0;
    unsigned long long e0 = block_excl_scan_u64(c0, s_scan, &t0);
    const int n_heads = (int)(t0 & 0xfffull), n_single = (int)((t0 >> 12) & 0xfffull), n_gw = (int)((t0 >> 24) & 0xfffull);
    const int n_k2 = (int)((t0 >> 36) & 0xfffull), n_k3 = (int)((t0 >> 48) & 0xfffull);
    const int n_pass = min(n_k3, n_heads);              // terminal states that ride along with a pair
    // SINGLES ON THE PAIR PATH: a staged single at offset o becomes a pair item with one dummy half — (single, dummy) when o
    // is even, (dummy, single) starting at o - 1 when it is odd — and is placed bank-aligned like a pair: it fills lanes
    // the pairs leave empty, and the one-state path (twice the shared-memory wavefronts per backup) is not run at all on
    // a cart-pole plane.  As many singles as the T item slots allow (each takes a whole slot instead of half of one).
    const int rest = n_gw + n_k2 + n_k3 - n_pass;
    const int n_conv = max(0, min(n_single, 2 * T - 2 * n_heads - n_single - rest - 1));
    const int n_left = n_single - n_conv + rest;        // states that share generic items, two each
    const int half = (n_left + 1) / 2;
    // Round 2: bank-pair class counts of the aligned items (pairs + converted singles), 10-bit counters
    unsigned long long c1 = 0, c2 = 0, c3 = 0;          // classes 0-5 | 6-11 | 12-15
    {
        int sr = (int)((e0 >> 12) & 0xfffull);          // staged singles before this thread
#pragma unroll
        for (int i = 0; i < KP; ++i) {
            if (cat[i] == kSingle) { if (sr >= n_conv) cat[i] = kWork + 16; ++sr; }   // kWork + 16: an unconverted single
            if (cat[i] == kHead || cat[i] == kSingle) {
                const unsigned c = (codes[i] >> 13) & 15u;
                if (c < 6) c1 += 1ull << (10 * c);
                else if (c < 12) c2 += 1ull << (10 * (c - 6));
                else c3 += 1ull << (10 * (c - 12));
            }
        }
    }
    unsigned long long t1, t2, t3;
    unsigned long long e1 = block_excl_scan_u64(c1, s_scan, &t1);
    unsigned long long e2 = block_excl_scan_u64(c2, s_scan, &t2);
    unsigned long long e3 = block_excl_scan_u64(c3, s_scan, &t3);
    // aligned items: lane = class, half-warp = how many items of that class came before; the generic items keep the last
    // half-warps to themselves
    const int hcap = max(1, min(q.hcap, (T - half) / 16));
    int place[KP];                                // aligned items: item slot, or -1 - stray rank; generic: leftover number j; passengers: pair number
    unsigned long long c5 = 0;                          // aligned items whose lane was taken in all hcap half-warps
    {
        int sr = (int)((e0 >> 12) & 0xfffull), gw = (int)((e0 >> 24) & 0xfffull), k2 = (int)((e0 >> 36) & 0xfffull), k3 = (int)((e0 >> 48) & 0xfffull);
#pragma unroll
        for (int i = 0; i < KP; ++i) {
            place[i] = 0;
            if (cat[i] == kHead || cat[i] == kSingle) {
                const unsigned c = (codes[i] >> 13) & 15u;
                int r;
                if (c < 6) { r = (int)((e1 >> (10 * c)) & 1023ull); e1 += 1ull << (10 * c); }
                else if (c < 12) { r = (int)((e2 >> (10 * (c - 6))) & 1023ull); e2 += 1ull << (10 * (c - 6)); }
                else { r = (int)((e3 >> (10 * (c - 12))) & 1023ull); e3 += 1ull << (10 * (c - 12)); }
                if (r < hcap) {
                    place[i] = r * 16 + (int)c;
                    s_occ[place[i]] = 1;
                } else {
                    place[i] = -1 - (int)c5;
                    c5 += 1ull;
                }
                if (cat[i] == kSingle) ++sr;
            } else if (cat[i] == kWork + 16) {
                place[i] = sr - n_conv; ++sr;                              // unconverted singles first
            } else if (cat[i] == kWork) {
                place[i] = n_single - n_conv + gw; ++gw;
            } else if (cat[i] == kK2) {
                place[i] = n_single - n_conv + n_gw + k2; ++k2;
            } else if (cat[i] == kK3) {
                place[i] = k3 < n_pass ? k3 : n_single - n_conv + n_gw + n_k2 + (k3 - n_pass);   // passenger of pair k3, or a leftover
                if (k3 < n_pass) cat[i] = kK3 + 16;                        // kK3 + 16: a passenger
                ++k3;
            }
        }
    }
    unsigned long long t5;
    const unsigned long long e5 = block_excl_scan_u64(c5, s_scan, &t5);   // (the barriers inside also publish s_occ)
    // free item slots in ascending order: generic items take them from the back (the last warp first), stray aligned items
    // the ones just before — the last half-warps are the emptiest, so a stray there rarely shares a bank with the rightful
    // owner of its class, and the strays of a plane cost one or two half-warps their conflict-free loads instead of five
    unsigned long long c6 = 0;
#pragma unroll
    for (int i = 0; i < kItemSlotsPer; ++i) {
        const int sl = tid * kItemSlotsPer + i;
        if (sl < T && !s_occ[sl]) c6 += 1ull;
    }
    unsigned long long t6;
    unsigned long long e6 = block_excl_scan_u64(c6, s_scan, &t6);
#pragma unroll
    for (int i = 0; i < kItemSlotsPer; ++i) {
        const int sl = tid * kItemSlotsPer + i;
        if (sl < T && !s_occ[sl]) { s_free[(int)e6] = (unsigned short)sl; e6 += 1ull; }
    }
    const int n_free = (int)t6;
    __syncthreads();
    // s_flag: where the code word of a state goes — 0 its own half, 1 nowhere (second state of a pair), 2 word 0 of the item
    // although the state sits in the second half (a single behind a dummy), 3 the state is a passenger
    {
        int pair_no = (int)(e0 & 0xfffull);            // pairs before this thread
#pragma unroll
        for (int i = 0; i < KP; ++i) {
            const int p = p0 + i;
            if (p >= P) continue;
            unsigned char flag = 0;
            if (cat[i] == kHead || cat[i] == kSingle) {
                int sl = place[i];
                if (sl < 0) sl = s_free[n_free - 1 - half - ((int)e5 + (-1 - sl))];
                if (cat[i] == kHead) {
                    s_dst[p] = (unsigned short)(sl * 2);
                    s_code[p] = (codes[i] & 0x07ffffffu) | kItemPair;                       // both halves valid
                    s_hslot[pair_no++] = (unsigned short)sl;
                } else if (((codes[i] >> 12) & 1u) == 0u) {
                    s_dst[p] = (unsigned short)(sl * 2);
                    s_code[p] = (codes[i] & 0x07ffffffu) | kItemPair | (1u << kItemKindShift);   // (single, dummy)
                } else {
                    s_dst[p] = (unsigned short)(sl * 2 + 1);
                    s_code[p] = ((codes[i] & 0x07ffffffu) - 0x1001u) | kItemPair | (2u << kItemKindShift);   // (dummy, single): one index, one offset back
                    flag = 2;
                }
            } else if (cat[i] == kTail) {
                flag = 1;
            } else if (cat[i] == kK3 + 16) {
                flag = 3;
            } else {
                const int j = place[i];
                const int item = j < half ? j : n_left - 1 - j;
                s_dst[p] = (unsigned short)(s_free[n_free - 1 - item] * 2 + (j < half ? 0 : 1));
            }
            s_flag[p] = flag;
        }
    }
    __syncthreads();
#pragma unroll
    for (int i = 0; i < KP; ++i) {
        const int p = p0 + i;
        if (p >= P) continue;
        if (cat[i] == kTail) s_dst[p] = (unsigned short)(s_dst[p - 1] + 1);
        if (cat[i] == kK3 + 16) {   // the second code word of pair item place[i] carries this terminal state
            const int sl = s_hslot[place[i]];
            stage[((size_t)(W >> 2) * T + sl) * 4 + (W & 3)] = kItemPair | (unsigned)p;
        }
    }
    __syncthreads();

    // ---- D. the row words of every state go to its place in the item array (staged in shared memory, stored coalesced)
    const int n4 = W / 4, n2 = (W % 4) / 2, n1 = W % 2;
    auto put = [&](int dst, int j, unsigned v) {   // word j of the state in half (dst & 1) of item slot (dst >> 1)
        const int jj = (dst & 1) * W + j;
        stage[((size_t)(jj >> 2) * T + (dst >> 1)) * 4 + (jj & 3)] = v;
    };
#pragma unroll
    for (int r = 0; r < KP; ++r) {
        const int t = tid + r * kItemThreads;
        if (t >= P) continue;
        const int flag = s_flag[t];
        if (flag == 3) continue;                           // passenger
        const int dst = s_dst[t];
        if (flag == 0) put(dst, 0, s_code[t]);
        else if (flag == 2) put(dst & ~1, 0, s_code[t]);
        {
            const uint4 v = *reinterpret_cast<const uint4*>(q.rows + (size_t)(s0 + t) * 16u);
            put(dst, 1, v.y); put(dst, 2, v.z); put(dst, 3, v.w);
        }
        for (int qq = 1; qq < n4; ++qq) {
            const uint4 v = *reinterpret_cast<const uint4*>(q.rows + (size_t)qq * 16u * (size_t)q.n_pad + (size_t)(s0 + t) * 16u);
            put(dst, 4 * qq, v.x); put(dst, 4 * qq + 1, v.y); put(dst, 4 * qq + 2, v.z); put(dst, 4 * qq + 3, v.w);
        }
        if (n2) {
            const uint2 v = *reinterpret_cast<const uint2*>(q.rows + (size_t)n4 * 16u * (size_t)q.n_pad + (size_t)(s0 + t) * 8u);
            put(dst, 4 * n4, v.x); put(dst, 4 * n4 + 1, v.y);
        }
        if (n1) put(dst, W - 1, *reinterpret_cast<const unsigned*>(q.rows + ((size_t)n4 * 16u + (size_t)n2 * 8u) * (size_t)q.n_pad + (size_t)(s0 + t) * 4u));
    }
    __syncthreads();
    {
        const uint4* src = reinterpret_cast<const uint4*>(stage);
        uint4* dst = reinterpret_cast<uint4*>(q.irows + (size_t)pl * (size_t)q.nq * (size_t)T * 16u);
        for (int i = tid; i < q.nq * T; i += kItemThreads) dst[i] = src[i];
    }
    if (tid == 0) {
        q.cells[pl].n_unstaged = s_un;
        atomicAdd(q.stats + 6, (unsigned long long)n_heads);
        atomicAdd(q.stats + 7, (unsigned long long)t5);   // aligned items outside their lane
        atomicAdd(q.stats + 8, (unsigned long long)n_conv);   // singles on the pair path
    }
}

// Pass 2 — one WARP per chunk of L consecutive state-planes, sequential over the chunk (the slot state of step i depends on
// step i-1): which slot holds which V-plane, which planes must be loaded before each step and whether that load can be
// issued one step ahead.  Works on the few cells per plane pass 1 found, not on states.
constexpr int kSlotWarps = 4;
__global__ void __launch_bounds__(kSlotWarps * 32) plane_slots_kernel(const PlanParams q) {
    __shared__ int s_slot_vp[kSlotWarps][kPlanMaxSlots];     // V-plane held by each slot (-1: none)
    __shared__ int s_slot_used[kSlotWarps][kPlanMaxSlots];   // last step that reads the slot
    __shared__ int s_cs[kSlotWarps][kPlanMaxCells * kPlanMaxOC];
    __shared__ unsigned s_early[kSlotWarps][kPlanMaxLoads], s_late[kSlotWarps][kPlanMaxLoads];
    const int lane = threadIdx.x & 31, wq = threadIdx.x >> 5;
    const int chunk = q.c_begin + blockIdx.x * kSlotWarps + wq;
    if (chunk >= q.c_end) return;
    const int pl0 = plan_chunk_begin(q, chunk);
    const int Lc = plan_chunk_begin(q, chunk + 1) - pl0;
    int* slot_vp = s_slot_vp[wq];
    int* slot_used = s_slot_used[wq];
    int* cs = s_cs[wq];
    unsigned* early = s_early[wq];
    unsigned* late = s_late[wq];
    for (int s = lane; s < kPlanMaxSlots; s += 32) { slot_vp[s] = -1; slot_used[s] = -1000; }
    __syncwarp();
    int noc_shift = 0;
    while ((1 << noc_shift) < q.noc) ++noc_shift;
    unsigned long long a_loads = 0, a_late = 0, a_fb = 0, a_live = 0, a_cells = 0;

    for (int i = 0; i < Lc; ++i) {
        const PlaneCells pc = q.cells[pl0 + i];
        const int K = pc.n_cells;
        const int T = K << noc_shift;                       // (cell, outer corner) pairs of this plane
        // resident corner planes keep their slot
        for (int m = lane; m < T; m += 32) {
            const int vp = pc.vp[m >> noc_shift] + q.ooff[m & (q.noc - 1)];
            int found = -1;
            for (int s = 0; s < q.NS; ++s)
                if (slot_vp[s] == vp) found = s;
            cs[m] = found;
            if (found >= 0) slot_used[found] = i;
        }
        __syncwarp();
        // allocate slots for the missing planes, one at a time (slot scan in parallel across the lanes)
        int n_early = 0, n_late = 0;
        unsigned bad = 0;                                   // cells that could not be staged (no slot left)
        for (int m0 = 0; m0 < T; m0 += 32) {
            const int mine_m = m0 + lane;
            unsigned todo = __ballot_sync(0xffffffffu, mine_m < T && cs[mine_m] < 0);
            while (todo) {
                const int m = m0 + __ffs(todo) - 1;
                todo &= todo - 1;
                const int k = m >> noc_shift;
                if ((bad >> k) & 1u) continue;
                const int vp = pc.vp[k] + q.ooff[m & (q.noc - 1)];
                int mine = -1, best_early = -1, best_late = -1;
                for (int s = lane; s < q.NS; s += 32) {
                    const int u = slot_used[s];
                    if (slot_vp[s] == vp && u == i) mine = s;      // allocated earlier in this step (another cell shares the plane)
                    if (u < i - 1 && best_early < 0) best_early = s;
                    if (u == i - 1 && best_late < 0) best_late = s;
                }
                const unsigned mm = __ballot_sync(0xffffffffu, mine >= 0);
                const unsigned me = __ballot_sync(0xffffffffu, best_early >= 0);
                const unsigned ml = __ballot_sync(0xffffffffu, best_late >= 0);
                int slot = -1, kind = 0;   // kind 1: early, 2: late
                if (mm) slot = __shfl_sync(0xffffffffu, mine, __ffs(mm) - 1);
                else if (me) { slot = __shfl_sync(0xffffffffu, best_early, __ffs(me) - 1); kind = i > 0 ? 1 : 2; }   // first plane of a chunk: late until stitched
                else if (ml) { slot = __shfl_sync(0xffffffffu, best_late, __ffs(ml) - 1); kind = 2; }
                if (slot < 0 || (kind && n_early + n_late >= kPlanMaxLoads)) {
                    bad |= 1u << k;
                } else {
                    if (lane == 0) {
                        cs[m] = slot;
                        if (kind) {
                            slot_vp[slot] = vp;
                            slot_used[slot] = i;
                            const unsigned e = ((unsigned)slot << 24) | (unsigned)vp;
                            if (kind == 1) early[n_early] = e;
                            else late[n_late] = e;
                        }
                    }
                    if (kind == 1) ++n_early;
                    else if (kind == 2) ++n_late;
                }
                __syncwarp();
            }
        }
        // outputs
        PlaneRec* rec = q.plan + pl0 + i;
        if (lane == 0) {
            rec->n_early = (unsigned char)n_early;
            rec->n_late = (unsigned char)n_late;
            rec->n_cells = (unsigned char)K;
            rec->flags = (unsigned char)bad;
            rec->pad[0] = rec->pad[1] = rec->pad[2] = 0u;
        }
        for (int t = lane; t < kPlanMaxCells * kPlanMaxOC; t += 32) {
            const int k = t / kPlanMaxOC, j = t - k * kPlanMaxOC;
            unsigned short v = 0;
            if (k < K && j < q.noc) {
                if ((bad >> k) & 1u) v = kPlanBadSlot;
                else v = (unsigned short)(((size_t)cs[(k << noc_shift) + j] * (size_t)q.pitch * 4u) >> 4);
            }
            rec->cs[k][j] = v;
        }
        for (int t = lane; t < n_early + n_late; t += 32) rec->loads[t] = t < n_early ? early[t] : late[t - n_early];
        // what plane_stitch_kernel works with: the slots the first step loads (all of its loads are late so far), and the
        // slots the last step reads or loads (slot_used == i: also the planes of a cell that was given up half-way)
        if (i == 0) {
            unsigned m[4] = {0u, 0u, 0u, 0u};
            for (int t = lane; t < n_early + n_late; t += 32) {
                const unsigned s = (t < n_early ? early[t] : late[t - n_early]) >> 24;
                m[s >> 5] |= 1u << (s & 31);
            }
#pragma unroll
            for (int w = 0; w < 4; ++w) m[w] = __reduce_or_sync(0xffffffffu, m[w]);
            if (lane < 4) q.chunk_slots[chunk].first[lane] = m[lane];
        }
        if (i == Lc - 1) {
            unsigned m[4] = {0u, 0u, 0u, 0u};
            for (int s = lane; s < q.NS; s += 32)
                if (slot_used[s] == i) m[s >> 5] |= 1u << (s & 31);
#pragma unroll
            for (int w = 0; w < 4; ++w) m[w] = __reduce_or_sync(0xffffffffu, m[w]);
            if (lane < 4) q.chunk_slots[chunk].last[lane] = m[lane];
        }
        a_loads += (unsigned long long)(n_early + n_late);
        a_late += (unsigned long long)n_late;
        a_fb += (unsigned long long)pc.n_unstaged;
        a_live += (unsigned long long)pc.n_unstaged;
        for (int k = 0; k < K; ++k) {
            a_live += pc.cnt[k];
            if ((bad >> k) & 1u) a_fb += pc.cnt[k];
            else a_cells += 1;
        }
        __syncwarp();
    }
    if (lane == 0) {
        atomicAdd(q.stats + 0, a_loads);
        atomicAdd(q.stats + 1, a_late);
        atomicAdd(q.stats + 2, a_fb);
        atomicAdd(q.stats + 3, a_live);
        atomicAdd(q.stats + 4, a_cells);
        atomicAdd(q.stats + 5, (unsigned long long)Lc);
    }
}

// Pass 3 — one WARP per CTA of the sweep, sequential over that CTA's chunks (the numbering of a chunk depends on the one
// before it): a chunk's first step loads every plane it reads, into slots numbered as if the chunk started cold.  A slot
// renumbering (a bijection: inside the chunk every load keeps its early / late kind) moves as many of those loads as
// possible into slots the CTA's previous chunk neither reads nor loads in its last step; the sweep issues them one step
// ahead, as inside a chunk.  The CTA's first chunk keeps its numbering and has no early loads there.
__device__ __forceinline__ int plan_rank(const unsigned (&m)[4], int s) {   // set bits of m below bit s
    int r = 0;
#pragma unroll
    for (int w = 0; w < 4; ++w) r += 32 * w + 32 <= s ? __popc(m[w]) : 32 * w < s ? __popc(m[w] & ((1u << (s - 32 * w)) - 1u)) : 0;
    return r;
}
__device__ __forceinline__ int plan_select(const unsigned (&m)[4], int j) {   // bit number of the j-th set bit of m
#pragma unroll
    for (int w = 0; w < 4; ++w) {
        unsigned x = m[w];
        const int c = __popc(x);
        if (j < c) {
            for (; j > 0; --j) x &= x - 1u;
            return 32 * w + __ffs(x) - 1;
        }
        j -= c;
    }
    return -1;
}
__global__ void __launch_bounds__(kSlotWarps * 32) plane_stitch_kernel(const PlanParams q) {
    constexpr int kPer = (kPlanMaxSlots + 31) / 32;
    const int lane = threadIdx.x & 31;
    const int b = blockIdx.x * kSlotWarps + (threadIdx.x >> 5);
    if (b >= q.grid) return;
    unsigned valid[4];
#pragma unroll
    for (int w = 0; w < 4; ++w) valid[w] = q.NS >= 32 * w + 32 ? 0xffffffffu : q.NS > 32 * w ? (1u << (q.NS - 32 * w)) - 1u : 0u;
    int perm[kPer];   // numbering of the previous chunk: slot lane + 32 w -> perm[w]
    int prev = -1;
    for (int ci = b; ci < q.n_chunks; ci += q.grid) {
        const int c = plan_chunk_at(q, ci);
        ChunkStitch* st = q.stitch + c;
        unsigned busy[4] = {0u, 0u, 0u, 0u};
        if (prev < 0) {
#pragma unroll
            for (int w = 0; w < kPer; ++w) perm[w] = lane + 32 * w;
        } else {
            const ChunkSlots cp = q.chunk_slots[prev], cc = q.chunk_slots[c];
#pragma unroll
            for (int w = 0; w < kPer; ++w) {
                const int s = lane + 32 * w;
                if (s < q.NS && ((cp.last[w] >> lane) & 1u)) busy[perm[w] >> 5] |= 1u << (perm[w] & 31);
            }
            unsigned fr[4];
#pragma unroll
            for (int w = 0; w < 4; ++w) {
                busy[w] = __reduce_or_sync(0xffffffffu, busy[w]);
                fr[w] = ~busy[w] & valid[w];
            }
            // planned order: the first step's loads, then the other slots; target order: free slots, then busy ones
            int n_t = 0, n_free = 0;
#pragma unroll
            for (int w = 0; w < 4; ++w) { n_t += __popc(cc.first[w] & valid[w]); n_free += __popc(fr[w]); }
#pragma unroll
            for (int w = 0; w < kPer; ++w) {
                const int s = lane + 32 * w;
                if (s >= q.NS) continue;
                const int r = plan_rank(cc.first, s);
                const int j = ((cc.first[w] >> lane) & 1u) ? r : n_t + (s - r);
                perm[w] = j < n_free ? plan_select(fr, j) : plan_select(busy, j - n_free);
            }
        }
        if (lane < 4) st->busy[lane] = busy[lane];
#pragma unroll
        for (int w = 0; w < kPer; ++w)
            if (lane + 32 * w < kPlanMaxSlots) st->perm[lane + 32 * w] = (unsigned char)perm[w];
        if (lane == 0) st->relabel = prev >= 0;
        prev = c;
    }
}

// Pass 4 — one CTA per chunk: apply plane_stitch_kernel's numbering to the chunk's slot offsets and load lists; the loads
// of the first step whose new slot the previous chunk does not touch become early (listed first).
constexpr int kRelabelThreads = 128;
__global__ void __launch_bounds__(kRelabelThreads) plane_relabel_kernel(const PlanParams q) {
    __shared__ unsigned char perm[kPlanMaxSlots];
    __shared__ unsigned busy[4];
    const int c = blockIdx.x, tid = threadIdx.x, lane = tid & 31;
    const ChunkStitch* st = q.stitch + c;
    if (!st->relabel) return;
    if (tid < kPlanMaxSlots) perm[tid] = st->perm[tid];
    if (tid < 4) busy[tid] = st->busy[tid];
    __syncthreads();
    const int pl0 = plan_chunk_begin(q, c);
    const int pl1 = plan_chunk_begin(q, c + 1);
    const unsigned unit = (unsigned)q.pitch / 4u;   // slot offset entry = slot * pitch * 4 / 16
    for (int pl = pl0; pl < pl1; ++pl) {
        PlaneRec* r = q.plan + pl;
        const unsigned hdr = *reinterpret_cast<const unsigned*>(r);
        const int K = (hdr >> 16) & 0xff, flags = hdr >> 24, n = (hdr & 0xff) + ((hdr >> 8) & 0xff);
        for (int t = tid; t < kPlanMaxCells * kPlanMaxOC; t += kRelabelThreads) {
            const int k = t / kPlanMaxOC, j = t % kPlanMaxOC;
            if (k < K && j < q.noc && !((flags >> k) & 1)) r->cs[k][j] = (unsigned short)(perm[r->cs[k][j] / unit] * unit);
        }
        if (pl > pl0) {
            for (int t = tid; t < n; t += kRelabelThreads) {
                const unsigned e = r->loads[t];
                r->loads[t] = ((unsigned)perm[e >> 24] << 24) | (e & 0xffffffu);
            }
        } else if (tid < 32) {
            constexpr int kPer = (kPlanMaxLoads + 31) / 32;
            unsigned e[kPer];
            bool early[kPer];
            unsigned me[kPer];
            int n_early = 0;
#pragma unroll
            for (int w = 0; w < kPer; ++w) {
                const int t = lane + 32 * w;
                e[w] = 0u;
                early[w] = false;
                if (t < n) {
                    const unsigned s = perm[r->loads[t] >> 24];
                    e[w] = (s << 24) | (r->loads[t] & 0xffffffu);
                    early[w] = !((busy[s >> 5] >> (s & 31)) & 1u);
                }
                me[w] = __ballot_sync(0xffffffffu, t < n && early[w]);
                n_early += __popc(me[w]);
            }
            __syncwarp();
            int before_e = 0;
#pragma unroll
            for (int w = 0; w < kPer; ++w) {
                const int t = lane + 32 * w;
                const int re = before_e + __popc(me[w] & ((1u << lane) - 1u));   // early loads before this one
                if (t < n) r->loads[early[w] ? re : n_early + (t - re)] = e[w];
                before_e += __popc(me[w]);
            }
            if (lane == 0) {
                r->n_early = (unsigned char)n_early;
                r->n_late = (unsigned char)(n - n_early);
                atomicAdd(q.stats + 1, 0ull - (unsigned long long)n_early);
            }
        }
        __syncthreads();
    }
}

// Layout probe: how many distinct successor cells of the outer dimensions does a state-plane of P states see
// (rows of ONE action, planes [0, n_planes) of a temporary table)?  1 when the dynamics are translation-invariant
// in the two fastest-stored dimensions.  out[0] += distinct cells, out[1] += planes with a live state.
__global__ void __launch_bounds__(kPlanThreads) plane_cells_probe_kernel(const unsigned char* rows, int P, int n_planes,
                                                                         unsigned long long* out) {
    __shared__ int htab[kPlanHash];
    __shared__ int overflow;
    const int tid = threadIdx.x;
    for (int pl = blockIdx.x; pl < n_planes; pl += gridDim.x) {
        if (tid < kPlanHash) htab[tid] = -1;
        if (tid == 0) overflow = 0;
        __syncthreads();
        for (int t = tid; t < P; t += kPlanThreads) {
            const int base = *reinterpret_cast<const int*>(rows + ((size_t)pl * P + t) * 16u);
            if (base < 0) continue;
            const int vp = base / P;
            int h = (int)(((unsigned)vp * 2654435761u) >> 27);
            bool ok = false;
            for (int probe = 0; probe < kPlanHash && !ok; ++probe) {
                const int old = atomicCAS(&htab[h], -1, vp);
                ok = old == -1 || old == vp;
                h = (h + 1) & (kPlanHash - 1);
            }
            if (!ok) overflow = 1;
        }
        __syncthreads();
        if (tid < 32) {
            const unsigned m = __ballot_sync(0xffffffffu, htab[tid] != -1);
            if (tid == 0 && m) {
                atomicAdd(out, (unsigned long long)(overflow ? 4 * kPlanHash : __popc(m)));
                atomicAdd(out + 1, 1ull);
            }
        }
        __syncthreads();
    }
}

}  // namespace pi
