// k_sgm.cu — K2: semi-global path aggregation (K3 — WTA / left-right check / sub-pixel — follows in k_wta.cu).
//
// No counterpart in the reference (SURVEY §0.2): this implements the frozen spec of DESIGN.md §3.3 (Hirschmueller 2008,
// fixed P1/P2), bit-exact against oracle/sva_oracle.c.
//
//   L_r(p,d) = C(p,d) + min(L_r(q,d), L_r(q,d-1)+P1, L_r(q,d+1)+P1, min_k L_r(q,k)+P2) - min_k L_r(q,k),  q = p - r
//   S = sum_r L_r (u16; C <= 4095 and P2 <= 4095 bound L by 8190 and S over 8 paths by 65520)
//
// Mapping: ONE WARP PER PATH LINE per direction.  A lane owns n = 2*NR consecutive disparities packed two per register
// (u16x2); the recurrence is DPX (VIADDMNMX.U16x2 / VIMNMX.U16x2), the d-1 / d+1 neighbours are one PRMT per register plus
// two warp shuffles for the lane edges, and min_k is a VIMNMX3 fold followed by one CREDUX.MIN.  Everything stays in
// registers along the path; C is streamed by cp.async (LDGSTS) into a per-warp ring of PF + 1 shared-memory stages, S is
// accumulated with fire-and-forget 64-bit REDs (packed u16x4 adds are carry-free by the bound above) into a zeroed volume.
// Diagonal paths use W lines of exactly H steps that wrap around the image edge and restart (L = C) where the predecessor
// is outside the image, so every line of a launch has the same length.
//
// Schedule for 8 paths (sva_run_sgm): four launches — the horizontal direction -> first, WRITING S with plain stores (so S is never
// zeroed), then <- accumulating with REDs like everything after it, then the three directions that sweep the rows downwards and the
// three that sweep upwards.  All lines of a row-sweeping launch advance one row per step, so a row's C and S lines are touched by all
// three directions while they are L2-resident (DRAM sees C once and S once per launch); when an image row of C + S is 768 KB or more
// the CTAs are additionally paced against the grid-wide minimum.  The single-direction horizontal launches have only H warps: <- runs
// on the second stream next to the first row-sweeping group where that group is not paced.  (Other groupings, several lines per warp
// and a last pass fused with K3 were measured and dropped: DESIGN.md §4.)
#include <algorithm>
#include <cstdio>
#include <cstdlib>

#include "sva_common.cuh"
#include "sva_vec.cuh"

#define SGM_INF2 0x7FFF7FFFu
constexpr size_t SGM_SMEM_PER_SM = 218 * 1024;  // ring space a resident wave may use per SM (228 KB minus the per-CTA reserve and the statics)
constexpr int SGM_WARPS_PER_SM = 46;            // marching warps per SM at 40 registers: two CTAs of 23 + 1 helper warp (warps are allocated in fours:
                                                // 2 x 24 x 32 x 40 registers fit the 64 K file, 2 x 28 do not)
constexpr int SGM_PF = 8;  // steps of prefetch in flight per warp; the ring has PF + 1 stages (the slot refilled at step s was last read at step s-1)

struct SgmParams {
    const uint16_t* C;
    uint16_t* S;
    int W, H, D;
    int ndirs;          // directions of this launch
    int dxs[8], dys[8];
    uint32_t p1p1, p2p2;
    int lanes;          // active lanes = D / (2*NR)
    unsigned int* pace_arrive;  // [pace_rounds] CTAs that finished round r (nullptr = no global pacing)
    unsigned int* pace_min;     // rounds finished by every CTA
    int pace_rounds, pace_window, march_warps;
    int diag_split;     // diagonals run the event-split march (launches that are not paced)
    int c_ds;           // 0: C is [H][W][D]; > 0: C is slice-major [D / c_ds][H][W][c_ds] (disparity slices gathered from several GPUs)
    int balanced;       // grid = m * SM count; warp w of CTA b handles direction w % ndirs, line b + grid * (w / ndirs)
    int ranged;         // 1: direction i contributes only its lines [line_lo[i], line_lo[i] + line_cnt[i]); warp w of CTA b takes the
    int line_lo[8], line_cnt[8];  //    (b + grid * w)-th line of the concatenated ranges (a launch cut to what is resident at once)
    // row-block pipeline across GPUs (sva_run_sgm_rows): a row-sweeping launch marches only image rows [row_y0, row_y0 + row_cnt) and
    // hands the state of every path line — L after the block's last row — to the GPU that owns the next rows
    int row_y0, row_cnt;
    const uint16_t* state_in;   // [3][W][D] (slot, line, disparity in the lane layout of S); nullptr where the block starts the sweep
    uint16_t* state_out;        // same shape; nullptr where the block ends the sweep
    int state_slot[8];          // slot of direction i of this launch
    uint32_t elem_bytes;        // sizeof(uint16_t), as a run-time value (see sgm_elem)
};

// one step of the recurrence for this lane's 2*NR disparities; L holds L(q,.) on entry and L(p,.) on exit
// EDGE_BIAS (every lane active): instead of replacing the missing d-1 / d+1 neighbour of the first / last disparity by
// +inf with two selects per step, the lane adds a per-lane P1 whose edge half is 0x7FFF (p1_up, p1_dn): the neighbour slot then holds a
// bounded real value (<= 8190), 8190 + 0x7FFF < 2^16 does not wrap and is larger than every real cost, so the minimum ignores it.
// BL > 0 (NR = 4): the block layout of VecBlk4 on BL lanes — registers 0,1 hold disparities 4l..4l+3, registers 2,3 hold 4BL+4l..4BL+4l+3,
// so each block has its own lane-edge neighbours (two rotations each way among the BL active lanes; disparities 4BL-1 | 4BL meet across
// lanes BL-1 | 0).  The range ends use the biased P1 of EDGE_BIAS: every rotation source is an active lane, so the stand-in is bounded.
template <int NR, bool EDGE_BIAS, int BL>
__device__ __forceinline__ void sgm_step(uint32_t (&L)[NR], const uint32_t (&Cc)[NR], uint32_t& mm, uint32_t& mp2, uint32_t p1p1, uint32_t p2p2,
                                         bool first_lane, bool last_lane, uint32_t p1_up, uint32_t p1_dn) {
    uint32_t dm[NR], dp[NR];  // values at d-1 / d+1 of register j
    if (BL > 0) {
        static_assert(BL == 0 || NR == 4, "block layout: 8 disparities per lane");
        const int lane = threadIdx.x & 31;
        const int prev = first_lane ? BL - 1 : lane - 1, next = last_lane ? 0 : lane + 1;  // (lanes beyond BL idle along; any source will do)
        const uint32_t a = __shfl_sync(0xffffffffu, L[1], prev), b = __shfl_sync(0xffffffffu, L[NR - 1], prev);
        const uint32_t c = __shfl_sync(0xffffffffu, L[0], next), d = __shfl_sync(0xffffffffu, L[NR - 2], next);
        const uint32_t up1 = first_lane ? a : b, dn0 = last_lane ? d : c;  // lane 0's a / lane BL-1's d: the other block's edge cell
        dm[0] = __byte_perm(a, L[0], 0x5432);  // lane 0: a stands in for the missing d-1 of disparity 0 (any real value: p1_up is biased)
        dp[0] = dm[1] = __byte_perm(L[0], L[1], 0x5432);
        dp[1] = __byte_perm(L[1], dn0, 0x5432);
        dm[NR - 2] = __byte_perm(up1, L[NR - 2], 0x5432);
        dp[NR - 2] = dm[NR - 1] = __byte_perm(L[NR - 2], L[NR - 1], 0x5432);
        dp[NR - 1] = __byte_perm(L[NR - 1], d, 0x5432);  // lane BL-1: d stands in for the missing d+1 of the last disparity (p1_dn is biased)
    } else {
        uint32_t up = __shfl_up_sync(0xffffffffu, L[NR - 1], 1);
        uint32_t dn = __shfl_down_sync(0xffffffffu, L[0], 1);
        if (!EDGE_BIAS) {
            if (first_lane) up = SGM_INF2;
            if (last_lane) dn = SGM_INF2;
            p1_up = p1p1; p1_dn = p1p1;
        }
        dm[0] = __byte_perm(up, L[0], 0x5432);
#pragma unroll
        for (int j = 1; j < NR; j++) dp[j - 1] = dm[j] = __byte_perm(L[j - 1], L[j], 0x5432);
        dp[NR - 1] = __byte_perm(L[NR - 1], dn, 0x5432);
    }
    uint32_t mloc = 0xFFFFFFFFu;
#pragma unroll
    for (int j = 0; j < NR; j++) {
        uint32_t t = __viaddmin_u16x2(dm[j], j == 0 ? p1_up : p1p1, L[j]);
        t = __viaddmin_u16x2(dp[j], j == NR - 1 ? p1_dn : p1p1, t);
        t = __vminu2(t, mp2);
        L[j] = Cc[j] + t - mm;  // both halves: t >= mm, no borrow; C + t - mm <= 8190, no carry
        mloc = __vminu2(mloc, L[j]);
    }
    const uint32_t m = __reduce_min_sync(0xffffffffu, min(mloc & 0xFFFFu, mloc >> 16));
    mm = m * 0x10001u;
    mp2 = mm + p2p2;
}

int sva_run_wta(sva_ctx* ctx, const uint16_t* vol);

// ---- how a warp moves its cells: per-lane cp.async (LDGSTS) into a ring of PF + 1 shared-memory stages, S accumulated by per-lane
// 64-bit REDs (every lane issues its own 4..16-byte piece; the TMA engine's bulk copies measured slower: DESIGN.md §4) -----------------
__host__ __device__ constexpr int sgm_warp_smem(const int nr, const int pf) { return (pf + 1) * 32 * 2 * nr * 2; }  // bytes per warp: the ring

// base + 2 * idx as ONE IMAD.WIDE on the (idle) FMA pipe.  Left to itself the compiler builds the 64-bit address of a u16 element from a
// 32-bit index with integer-ALU instructions (IADD3 / IADD3.X carry chains, or LEA + LEA.HI.X when it sees the constant 2) — on the pipe that
// bounds the march.  `two` is the element size read from the kernel parameters, so that it stays a multiplication.
__device__ __forceinline__ const uint16_t* sgm_elem(const uint16_t* base, const uint32_t idx, const uint32_t two) {
    unsigned long long a;
    asm("mad.wide.u32 %0, %1, %2, %3;" : "=l"(a) : "r"(idx), "r"(two), "l"((unsigned long long)(uintptr_t)base));
    return (const uint16_t*)(uintptr_t)a;
}

template <int NR, int PF, bool FULL, bool STORE, int BL>
struct SgmPipe {
    static constexpr int NS = PF + 1, NV = 2 * NR, STAGE = 32 * NV * 2;
    using V = typename VecSel<NR, BL>::type;
    // Cursors are CELL indices times D, the same in every lane (warp-uniform: the compiler keeps them on the uniform datapath); what differs per
    // lane is folded into the base pointers.
    const uint16_t* C;  // cost volume + this lane's offset
    uint16_t* S;        // aggregation volume + this lane's offset
    uint32_t ring;      // this lane's bytes inside stage 0
    uint32_t two;
    bool active;
    __device__ __forceinline__ void init(const SgmParams& q, const uint32_t warp_base, const int lane, const bool active_) {
        constexpr int LANE_ELEMS = BL ? 4 : NV;
        const int le = lane * LANE_ELEMS;
        // slice-major cost volume: a lane's cells never straddle a slice (c_ds % NV == 0)
        const size_t lane_c = q.c_ds > 0 ? (size_t)(le / q.c_ds) * q.H * q.W * q.c_ds + le % q.c_ds : (size_t)le;
        C = q.C + lane_c;
        S = q.S + le;
        ring = warp_base + lane * (BL ? 8 : 4 * NR);
        two = q.elem_bytes;
        active = active_;
    }
    // start the copy of the cell at element index `ic` of C into stage `slot`
    __device__ __forceinline__ void fill(const int slot, const uint32_t ic) const {
        if (active) V::cp_async(ring + slot * STAGE, sgm_elem(C, ic, two));
    }
    __device__ __forceinline__ void fill_end() const { cp_async_commit(); }
    // the cell of step t (stage t % NS) -> registers
    __device__ __forceinline__ void take(const int slot, uint32_t (&Cc)[NR]) const {
        cp_async_wait<PF - 1>();
#pragma unroll
        for (int j = 0; j < NR; j++) Cc[j] = SGM_INF2;
        if (active) V::lds(ring + slot * STAGE, Cc);
    }
    // L of the cell just computed -> the cell at element index `is` of S
    __device__ __forceinline__ void emit(const uint32_t is, const uint32_t (&L)[NR]) const {
        uint16_t* dst = const_cast<uint16_t*>(sgm_elem(S, is, two));
        if (active) {
            if (STORE) V::store(dst, L); else V::red(dst, L);
        }
    }
};

// ---- the accumulate march: specialised at compile time on DIAG (wrap / restart logic only for diagonals), FULL (all 32 lanes
// active: no predicates) and STORE (plain store vs RED), running 32-bit element cursors instead of recomputed cell indices.
template <int NR, int PF, bool FULL, bool DIAG, bool STORE, int BL>
__device__ __forceinline__ void sgm_acc_march(const SgmParams& q, const int dx, const int dy, const int line, const int lane, const uint32_t warp_smem,
                                              const int bar_threads, volatile int* s_pace /* [0] rounds finished by this CTA, [1] rounds finished by every CTA */,
                                              const bool leader) {
    using Pipe = SgmPipe<NR, PF, FULL, STORE, BL>;
    constexpr int NS = Pipe::NS, NV = 2 * NR, LANE_ELEMS = BL ? 4 : NV;
    const int W = q.W, H = q.H, D = q.D;
    const int len = dy == 0 ? W : H;
    const int x0 = dy == 0 ? (dx > 0 ? 0 : W - 1) : line, y0 = dy == 0 ? line : (dy > 0 ? 0 : H - 1);
    // Cursors are 32-bit ELEMENT indices into the volumes (W*H*D < 2^32; the 64-bit address is one IMAD.WIDE on the FMA pipe), and
    // a diagonal's wrap at the image edge is a countdown instead of two coordinate compares: the recurrence saturates the integer
    // ALU pipe, so every ALU instruction shaved off the cursor bookkeeping is time.
    const uint32_t dstep = (uint32_t)((dy * W + dx) * D), wrapfix = (uint32_t)(-dx * W * D);
    const uint32_t start = (uint32_t)(((long long)y0 * W + x0) * D);
    // the cost volume may be slice-major: same walk, pixel stride c_ds (the lane's slice offset is part of the pipe's base pointer)
    const int cds = q.c_ds > 0 ? q.c_ds : D;
    const uint32_t dstep_c = (uint32_t)((dy * W + dx) * cds), wrapfix_c = (uint32_t)(-dx * W * cds);
    const uint32_t start_c = (uint32_t)(((long long)y0 * W + x0) * cds);
    uint32_t ic = start_c, is = start;                // prefetch cursor (C), accumulate cursor (S)
    int cc = dx > 0 ? W - x0 : x0 + 1, cs = cc;       // steps until each cursor leaves the image sideways
    const bool active = FULL || lane < q.lanes;
    const bool first_lane = lane == 0, last_lane = FULL ? lane == 31 : lane == q.lanes - 1;
    const uint32_t p1_up = first_lane ? (q.p1p1 & 0xFFFF0000u) | 0x7FFFu : q.p1p1, p1_dn = last_lane ? (q.p1p1 & 0x0000FFFFu) | 0x7FFF0000u : q.p1p1;
    Pipe pipe;
    pipe.init(q, warp_smem, lane, active);
    auto adv = [&](uint32_t& i, int& cnt, const uint32_t step, const uint32_t fix) -> bool {
        i += step;
        if (DIAG) {
            if (--cnt == 0) { cnt = W; i += fix; return true; }
        }
        return false;
    };
#pragma unroll
    for (int u = 0; u < PF; u++) {
        if (u < len) { pipe.fill(u, ic); adv(ic, cc, dstep_c, wrapfix_c); }
        pipe.fill_end();
    }
    uint32_t L[NR];
#pragma unroll
    for (int j = 0; j < NR; j++) L[j] = 0;
    uint32_t mm = 0, mp2 = q.p2p2;
    bool restart = false;  // step 0 starts from L = 0, mm = 0, which yields L = C
    auto step = [&](const int slot, const int refill_slot, const bool refill) {
        uint32_t Cc[NR];
        pipe.take(slot, Cc);
        if (refill) { pipe.fill(refill_slot, ic); adv(ic, cc, dstep_c, wrapfix_c); }
        pipe.fill_end();
        if (DIAG && restart) {
#pragma unroll
            for (int j = 0; j < NR; j++) L[j] = 0;
            mm = 0; mp2 = q.p2p2;
        }
        sgm_step<NR, FULL, BL>(L, Cc, mm, mp2, q.p1p1, q.p2p2, first_lane, last_lane, p1_up, p1_dn);
        pipe.emit(is, L);
        restart = adv(is, cs, dstep, wrapfix);
    };
    int s0 = 0;
    for (; s0 + NS + PF <= len; s0 += NS) {
        // keep the row-sweeping warps of this CTA in step (one named barrier per ring round): directions that sweep the rows in the
        // same order then touch the C and S lines they share within microseconds of each other, i.e. while they are in L2
        if (bar_threads) {
            asm volatile("bar.sync 1, %0;" ::"r"(bar_threads) : "memory");
            if (s_pace) {
                // global pacing (asynchronous): the helper warp publishes this CTA's progress and mirrors the grid-wide minimum into
                // shared memory; a CTA that is more than pace_window rounds ahead of the slowest one naps.  Bounded spin: never hangs.
                const int round = s0 / NS;
                if (leader && lane == 0) s_pace[0] = round;
                for (int spin = 0; spin < 4096 && round > s_pace[1] + q.pace_window; spin++) __nanosleep(128);
            }
        }
#pragma unroll
        for (int u = 0; u < NS; u++) step(u, (u + PF) % NS, true);
    }
    if (s_pace && leader && lane == 0) s_pace[0] = s0 / NS;  // all paced rounds done (lets the helper warp finish)
    for (int s = s0; s < len; s++) step(s % NS, (s + PF) % NS, s + PF < len);
}

// Diagonal march for ONE line per warp, split at the wrap events.  A diagonal leaves the image sideways once every W steps; the
// prefetch cursor does so PF steps before the accumulate cursor.  Between two such events nothing special happens, so the step body
// carries no wrap / restart logic at all (in the generic march that logic is ~8 predicated integer instructions per step on a kernel
// bound by the integer pipe): whole ring rounds of NS steps run unrolled, the few steps around an event run one at a time.  The wrap
// step is a per-line constant, i.e. warp-uniform here.  The CTA barrier / pacing rhythm (every NS steps, same step indices in every
// warp) is kept, so the warps of a CTA still meet the same number of times.
template <int NR, int PF, bool FULL, bool STORE, int BL>
__device__ __forceinline__ void sgm_acc_march_diag32(const SgmParams& q, const int dx, const int dy, const int line, const int lane,
                                                     const uint32_t warp_smem, const int bar_threads, volatile int* s_pace, const bool leader) {
    using Pipe = SgmPipe<NR, PF, FULL, STORE, BL>;
    constexpr int NS = Pipe::NS, NV = 2 * NR, LANE_ELEMS = BL ? 4 : NV;
    const int W = q.W, H = q.H, D = q.D;
    const int len = H;
    const int x0 = line, y0 = dy > 0 ? 0 : H - 1;
    const uint32_t dstep = (uint32_t)((dy * W + dx) * D), wrapfix = (uint32_t)(-dx * W * D);
    const uint32_t start = (uint32_t)(((long long)y0 * W + x0) * D);
    const int cds = q.c_ds > 0 ? q.c_ds : D;
    const uint32_t dstep_c = (uint32_t)((dy * W + dx) * cds), wrapfix_c = (uint32_t)(-dx * W * cds);
    const uint32_t start_c = (uint32_t)(((long long)y0 * W + x0) * cds);
    uint32_t ic = start_c, is = start;
    const bool active = FULL || lane < q.lanes;
    const bool first_lane = lane == 0, last_lane = FULL ? lane == 31 : lane == q.lanes - 1;
    const uint32_t p1_up = first_lane ? (q.p1p1 & 0xFFFF0000u) | 0x7FFFu : q.p1p1, p1_dn = last_lane ? (q.p1p1 & 0x0000FFFFu) | 0x7FFF0000u : q.p1p1;
    Pipe pipe;
    pipe.init(q, warp_smem, lane, active);
    int wc = dx > 0 ? W - x0 : x0 + 1;  // the prefetch cursor wraps after this many advances ...
    int ws = wc;                        // ... the accumulate cursor after this many (then every W more)
    int adv_c = 0;
#pragma unroll
    for (int u = 0; u < PF; u++) {
        if (u < len) {
            pipe.fill(u, ic);
            ic += dstep_c;
            if (++adv_c == wc) { ic += wrapfix_c; wc += W; }
        }
        pipe.fill_end();
    }
    uint32_t L[NR];
#pragma unroll
    for (int j = 0; j < NR; j++) L[j] = 0;
    uint32_t mm = 0, mp2 = q.p2p2;
    auto step = [&](const int slot, const int refill_slot, const bool refill) {
        uint32_t Cc[NR];
        pipe.take(slot, Cc);
        if (refill) { pipe.fill(refill_slot, ic); ic += dstep_c; }
        pipe.fill_end();
        sgm_step<NR, FULL, BL>(L, Cc, mm, mp2, q.p1p1, q.p2p2, first_lane, last_lane, p1_up, p1_dn);
        pipe.emit(is, L);
        is += dstep;
    };
    int s = 0, slot = 0, round = 0;  // slot == s % NS throughout
    while (s < len) {
        // last step before the next event: the prefetch cursor has advanced PF + s + 1 times after step s (while it refills)
        const int e_c = wc - PF - 1, e_s = ws - 1;
        const int e = min(len - 1, min(e_c, e_s));
        while (s <= e) {
            const bool paced = slot == 0 && s + NS + PF <= len;
            if (paced && bar_threads) {
                asm volatile("bar.sync 1, %0;" ::"r"(bar_threads) : "memory");
                if (s_pace) {
                    if (leader && lane == 0) s_pace[0] = round;
                    for (int spin = 0; spin < 4096 && round > s_pace[1] + q.pace_window; spin++) __nanosleep(128);
                }
            }
            if (paced) round++;
            if (paced && s + NS - 1 <= e) {  // a whole ring round without an event: every step refills
#pragma unroll
                for (int u = 0; u < NS; u++) step(u, (u + PF) % NS, true);
                s += NS;
            } else {
                const int rs = slot + PF >= NS ? slot + PF - NS : slot + PF;
                step(slot, rs, s + PF < len);
                s++;
                slot = slot + 1 == NS ? 0 : slot + 1;
            }
        }
        if (e == e_c) { ic += wrapfix_c; wc += W; }
        if (e == e_s) {  // the next cell starts a fresh path: L = C
            is += wrapfix; ws += W;
#pragma unroll
            for (int j = 0; j < NR; j++) L[j] = 0;
            mm = 0; mp2 = q.p2p2;
        }
    }
    if (s_pace && leader && lane == 0) s_pace[0] = round;  // all paced rounds done (lets the helper warp finish)
}

// Row-block march (dy != 0): the generic march over image rows [row_y0, row_y0 + row_cnt) only.  A line that was already under way
// above (below) the block continues from the L its previous owner stored; its minimum is recomputed from that L.  A line whose
// predecessor cell lies outside the image at the block's first row (the sweep's first row, or a diagonal that has just wrapped) starts
// fresh exactly as in the whole-frame march.  Column of line x0 after t rows: (x0 + dx * t) mod W.
template <int NR, int PF, bool FULL, bool STORE, int BL>
__device__ __forceinline__ void sgm_rows_march(const SgmParams& q, const int dx, const int dy, const int slot_of_dir, const int line, const int lane,
                                               const uint32_t warp_smem, const int bar_threads, volatile int* s_pace, const bool leader) {
    using Pipe = SgmPipe<NR, PF, FULL, STORE, BL>;
    using V = typename VecSel<NR, BL>::type;
    constexpr int NS = Pipe::NS, NV = 2 * NR, LANE_ELEMS = BL ? 4 : NV;
    const int W = q.W, H = q.H, D = q.D;
    const int len = q.row_cnt;
    const int ya = dy > 0 ? q.row_y0 : q.row_y0 + q.row_cnt - 1;  // first row of the block in sweep order
    const int t = dy > 0 ? ya : H - 1 - ya;                        // rows the line has already crossed
    int xa = (int)(((long long)line + (long long)dx * t) % W);
    if (xa < 0) xa += W;
    const uint32_t dstep = (uint32_t)((dy * W + dx) * D), wrapfix = (uint32_t)(-dx * W * D);
    const uint32_t start = (uint32_t)(((long long)ya * W + xa) * D);
    uint32_t ic = start, is = start;
    int cc = dx > 0 ? W - xa : (dx < 0 ? xa + 1 : 0x7FFFFFFF), cs = cc;  // steps until each cursor leaves the image sideways
    const bool active = FULL || lane < q.lanes;
    const bool first_lane = lane == 0, last_lane = FULL ? lane == 31 : lane == q.lanes - 1;
    const uint32_t p1_up = first_lane ? (q.p1p1 & 0xFFFF0000u) | 0x7FFFu : q.p1p1, p1_dn = last_lane ? (q.p1p1 & 0x0000FFFFu) | 0x7FFF0000u : q.p1p1;
    Pipe pipe;
    pipe.init(q, warp_smem, lane, active);
    auto adv = [&](uint32_t& i, int& cnt) -> bool {
        i += dstep;
        if (--cnt == 0) { cnt = W; i += wrapfix; return true; }
        return false;
    };
#pragma unroll
    for (int u = 0; u < PF; u++) {
        if (u < len) { pipe.fill(u, ic); adv(ic, cc); }
        pipe.fill_end();
    }
    const size_t state_at = ((size_t)slot_of_dir * W + line) * D + lane * LANE_ELEMS;
    const bool fresh = t == 0 || (dx > 0 && xa == 0) || (dx < 0 && xa == W - 1) || q.state_in == nullptr;
    uint32_t L[NR];
    uint32_t mm = 0, mp2 = q.p2p2;
#pragma unroll
    for (int j = 0; j < NR; j++) L[j] = 0;
    if (!fresh) {  // warp-uniform: t, xa and the pointer are per line
#pragma unroll
        for (int j = 0; j < NR; j++) L[j] = SGM_INF2;
        if (active) V::load(q.state_in + state_at, L);
        uint32_t mloc = L[0];
#pragma unroll
        for (int j = 1; j < NR; j++) mloc = __vminu2(mloc, L[j]);
        mm = __reduce_min_sync(0xffffffffu, min(mloc & 0xFFFFu, mloc >> 16)) * 0x10001u;
        mp2 = mm + q.p2p2;
    }
    bool restart = false;
    auto step = [&](const int slot, const int refill_slot, const bool refill) {
        uint32_t Cc[NR];
        pipe.take(slot, Cc);
        if (refill) { pipe.fill(refill_slot, ic); adv(ic, cc); }
        pipe.fill_end();
        if (restart) {
#pragma unroll
            for (int j = 0; j < NR; j++) L[j] = 0;
            mm = 0; mp2 = q.p2p2;
        }
        sgm_step<NR, FULL, BL>(L, Cc, mm, mp2, q.p1p1, q.p2p2, first_lane, last_lane, p1_up, p1_dn);
        pipe.emit(is, L);
        restart = adv(is, cs);
    };
    int s0 = 0;
    for (; s0 + NS + PF <= len; s0 += NS) {
        if (bar_threads) {  // same CTA rhythm and global pacing as the whole-frame march
            asm volatile("bar.sync 1, %0;" ::"r"(bar_threads) : "memory");
            if (s_pace) {
                const int round = s0 / NS;
                if (leader && lane == 0) s_pace[0] = round;
                for (int spin = 0; spin < 4096 && round > s_pace[1] + q.pace_window; spin++) __nanosleep(128);
            }
        }
#pragma unroll
        for (int u = 0; u < NS; u++) step(u, (u + PF) % NS, true);
    }
    if (s_pace && leader && lane == 0) s_pace[0] = s0 / NS;
    for (int s = s0; s < len; s++) step(s % NS, (s + PF) % NS, s + PF < len);
    if (q.state_out && active) V::store(q.state_out + state_at, L);
}

// g-th line of the concatenated per-direction ranges of a ranged launch
__device__ __forceinline__ bool sgm_ranged_line(const SgmParams& q, int g, int& dir, int& line) {
    for (int i = 0; i < q.ndirs; i++) {
        if (g < q.line_cnt[i]) { dir = i; line = q.line_lo[i] + g; return true; }
        g -= q.line_cnt[i];
    }
    return false;
}

// 40 registers: 48 resident warps per SM (e.g. two 22-warp CTAs of a paced c4 launch) must fit the 64 K register file
template <int NR, int PF, bool FULL, bool STORE, int BL, bool ROWS>
__global__ void __maxnreg__(40)
k_sgm_acc(SgmParams q) {
    constexpr int RING_BYTES = sgm_warp_smem(NR, PF);
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31;
    const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0);  // the same value, marked warp-uniform for the compiler: line, direction and
                                                                     // the cell cursors derived from it then live on the uniform datapath
    __shared__ volatile int s_pace[2];
    if (q.pace_arrive) {
        if (threadIdx.x == 0) { s_pace[0] = 0; s_pace[1] = 0; }
        __syncthreads();
        if (warp == q.march_warps) {
            // helper warp: all global pacing traffic happens here, off the marching warps' critical path.  arrive[r] counts the CTAs
            // that finished round r; whoever arrives last advances the grid-wide minimum.
            if (lane == 0) {
                int published = 0;
                for (int it = 0; it < (1 << 22) && published < q.pace_rounds; it++) {
                    const int r = s_pace[0];
                    for (; published < r; published++) {
                        unsigned int old = atomicAdd(q.pace_arrive + published, 1u);
                        if (old == gridDim.x - 1) { asm volatile("st.relaxed.gpu.global.u32 [%0], %1;" ::"l"(q.pace_min), "r"(published + 1) : "memory"); }
                    }
                    unsigned int g;
                    asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(g) : "l"(q.pace_min) : "memory");
                    s_pace[1] = (int)g;
                    __nanosleep(1000);
                }
            }
            return;
        }
    }
    int dir = 0, line = 0;
    if (q.ranged) {
        if (!sgm_ranged_line(q, q.balanced ? blockIdx.x + gridDim.x * warp : blockIdx.x * q.march_warps + warp, dir, line)) return;
    } else if (q.balanced) {  // every CTA carries the same mix of directions and every SM the same number of CTAs -> all lines advance at the same rate
        dir = warp % q.ndirs;
        line = blockIdx.x + gridDim.x * (warp / q.ndirs);
    } else {
        dir = blockIdx.x % q.ndirs; line = (blockIdx.x / q.ndirs) * q.march_warps + warp;
    }
    const int dx = q.dxs[dir], dy = q.dys[dir];
    const int nlines = dy == 0 ? q.H : q.W;
    if (line >= nlines) return;
    const uint32_t ring = smem_u32(smem_raw) + warp * RING_BYTES;  // this warp's stages
    int bar_threads = 0;
    bool leader = false;
    if (q.balanced && dy != 0) {  // threads of this CTA that march down/up the rows (all do the same number of rounds)
        int first = -1;
        for (int w = 0; w < q.march_warps; w++) {
            bool marches;
            if (q.ranged) {
                int d_ = 0, l_ = 0;
                marches = sgm_ranged_line(q, blockIdx.x + gridDim.x * w, d_, l_) && q.dys[d_] != 0;
            } else marches = q.dys[w % q.ndirs] != 0 && (int)(blockIdx.x + gridDim.x * (w / q.ndirs)) < q.W;
            if (marches) { bar_threads += 32; if (first < 0) first = w; }
        }
        leader = warp == first;
    }
    volatile int* pace = (q.pace_arrive && bar_threads) ? s_pace : nullptr;
    if (ROWS) {  // row-sweeping directions only (the host never puts a horizontal one into a ROWS launch)
        sgm_rows_march<NR, PF, FULL, STORE, BL>(q, dx, dy, q.state_slot[dir], line, lane, ring, bar_threads, pace, leader);
        return;
    }
    if (dx != 0 && dy != 0) {
        if (q.diag_split) sgm_acc_march_diag32<NR, PF, FULL, STORE, BL>(q, dx, dy, line, lane, ring, bar_threads, pace, leader);
        else sgm_acc_march<NR, PF, FULL, true, STORE, BL>(q, dx, dy, line, lane, ring, bar_threads, pace, leader);
    } else sgm_acc_march<NR, PF, FULL, false, STORE, BL>(q, dx, dy, line, lane, ring, bar_threads, pace, leader);
}

// Row-sweeping launches are paced when one image row of C + S is 768 KB or more (SVA_SGM_PACE pins the choice).
static bool sgm_paced(const sva_ctx* ctx, const SgmParams& q) {
    return ctx->tune_sgm_pace < 0 ? (size_t)q.W * q.D * 4 >= 768 * 1024 : ctx->tune_sgm_pace != 0;
}

// path lines one launch can keep resident at once: the marching warps per SM, or the rings that fit its shared memory
static int sgm_resident_lines(const sva_ctx* ctx, int nr) {
    return ctx->sm_count * std::min(SGM_WARPS_PER_SM, (int)(SGM_SMEM_PER_SM / sgm_warp_smem(nr, SGM_PF)));
}

template <int NR, int PF, bool FULL, bool STORE, int BL, bool ROWS = false>
static int launch_acc(sva_ctx* ctx, const SgmParams& q, const char* name) {
    constexpr size_t RING_BYTES = sgm_warp_smem(NR, PF);  // per warp
    constexpr int FALLBACK_WARPS = 8;
    int nlines = 0;
    for (int i = 0; i < q.ndirs; i++) nlines = std::max(nlines, q.dys[i] == 0 ? q.H : q.W);
    int warps = FALLBACK_WARPS, grid = div_up(nlines, FALLBACK_WARPS) * q.ndirs;
    SgmParams qq = q;
    qq.balanced = 0;
    // one wave of identical CTAs: m CTAs per SM, as few warps per CTA as cover all lines (every CTA the same mix of directions, every SM
    // the same number of CTAs, so all lines advance at the same rate); launches too large for one wave fall back to 8-warp CTAs
    int total = 0;
    for (int i = 0; i < q.ndirs; i++) total += q.line_cnt[i];
    for (int m = 1; m <= 8; m++) {
        const int g = ctx->sm_count * m;
        const int w = q.ranged ? div_up(total, g) : div_up(nlines, g) * q.ndirs;  // lines per direction per CTA x directions
        const size_t smem_cap = q.ranged ? SGM_SMEM_PER_SM : 200 * 1024;
        const int wmax = q.ranged ? 31 : 32;  // a ranged launch is always paced: leave room for the helper warp
        if (w <= wmax && (size_t)w * RING_BYTES * m <= smem_cap && w * 32 * m <= 2048) { warps = w; grid = g; qq.balanced = 1; break; }
    }
    if (q.ranged && !qq.balanced) grid = div_up(total, FALLBACK_WARPS);
    const size_t smem = (size_t)warps * RING_BYTES;
    SVA_CUDA_OK(ctx, cudaFuncSetAttribute(k_sgm_acc<NR, PF, FULL, STORE, BL, ROWS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    SVA_CUDA_OK(ctx, cudaFuncSetAttribute(k_sgm_acc<NR, PF, FULL, STORE, BL, ROWS>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    qq.march_warps = warps;
    qq.pace_arrive = nullptr;
    int threads = warps * 32;
    bool n_vert = false;
    for (int i = 0; i < q.ndirs; i++) n_vert = n_vert || q.dys[i] != 0;
    if (qq.balanced && sgm_paced(ctx, q) && q.ndirs > 1 && n_vert && q.W >= grid && warps < 32) {
        // global pacing needs every CTA resident (the grid is one balanced wave by construction; check the occupancy anyway)
        int per_sm = 0;
        SVA_CUDA_OK(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_sgm_acc<NR, PF, FULL, STORE, BL, ROWS>, threads + 32, smem));
        if (getenv("SVA_DEBUG")) fprintf(stderr, "[sva] sgm_acc NR=%d ndirs=%d grid=%d threads=%d smem=%zu per_sm=%d\n", NR, q.ndirs, grid, threads + 32, smem, per_sm);
        if ((long long)per_sm * ctx->sm_count >= grid) {
            const int rounds = ((ROWS ? q.row_cnt : q.H) - PF) / (PF + 1);
            if (rounds > ctx->tune_sgm_pace_window) {
                SVA_TRY(ctx->reserve(ctx->pace_buf, ((size_t)rounds + 16) * sizeof(unsigned int)));
                SVA_CUDA_OK(ctx, cudaMemsetAsync(ctx->pace_buf.p, 0, ((size_t)rounds + 16) * sizeof(unsigned int), ctx->stream));
                qq.pace_min = ctx->pace_buf.as<unsigned int>();
                qq.pace_arrive = qq.pace_min + 16;
                qq.pace_rounds = rounds;
                qq.pace_window = ctx->tune_sgm_pace_window;
                threads += 32;  // the helper warp
            }
        }
    }
    // measured: the event-split diagonal march gains 6.6 % on unpaced launches (c1: 0.279 -> 0.261 ms) and nothing on paced ones (c2 / c4
    // move at the pace of the grid-wide minimum), where the generic march is kept
    qq.diag_split = qq.pace_arrive == nullptr;
    {
        // timing label = the kernel's symbol as ncu prints it + "/" + what this launch carries
        char sym[96];
        snprintf(sym, sizeof sym, "k_sgm_acc<%d, %d, %d, %d, %d, %d>/%s%s", NR, PF, (int)FULL, (int)STORE, BL, (int)ROWS, name, q.ranged && q.dys[0] != 0 ? "_ranged" : "");
        LaunchScope ls(ctx, ctx->intern(sym));
        k_sgm_acc<NR, PF, FULL, STORE, BL, ROWS><<<grid, threads, smem, ctx->stream>>>(qq);
    }
    SVA_CUDA_OK(ctx, cudaGetLastError());
    return SVA_OK;
}

// the directions q.dxs / q.dys in ONE launch; store = plain stores (a single direction that initialises S) instead of REDs
template <int NR>
static int launch_dirs_nr(sva_ctx* ctx, const SgmParams& q, bool store) {
    const bool full = q.lanes == 32;
    // what the launch carries: row-sweeping directions (they share C and S lines in L2: the launch streams C once and read-modify-writes S
    // once), horizontal directions (-> and <- cannot share: each streams C and S), or a mix (4 paths)
    bool any_v = false, any_h = false;
    for (int i = 0; i < q.ndirs; i++) { any_v = any_v || q.dys[i] != 0; any_h = any_h || q.dys[i] == 0; }
    static const char* const cnt[9] = {"0", "1", "2", "3", "4", "5", "6", "7", "8"};
    const std::string what = std::string(store ? "store_" : "red_") + (any_v && any_h ? "mixed" : any_v ? (q.dys[0] > 0 ? "down" : "up") : "horizontal") + cnt[q.ndirs];
    const char* nm = ctx->intern(what);
    if (q.row_cnt > 0 && q.dys[0] != 0) {  // a row block of a row-sweeping group (REDs only, contiguous volume)
        if (store || q.c_ds != 0) return ctx->fail(SVA_ERR_BAD_ARG, "internal: row-block launches accumulate into a contiguous volume");
        if constexpr (NR == 4) {
            if (q.lanes == 32) return launch_acc<NR, SGM_PF, true, false, 32, true>(ctx, q, nm);
            if (q.lanes == 24) return launch_acc<NR, SGM_PF, false, false, 24, true>(ctx, q, nm);
        }
        return full ? launch_acc<NR, SGM_PF, true, false, 0, true>(ctx, q, nm) : launch_acc<NR, SGM_PF, false, false, 0, true>(ctx, q, nm);
    }
    if constexpr (NR == 4) {  // D = 256 / 192 on a contiguous volume: the block layout (whole-sector copies and REDs)
        if (q.c_ds == 0) {
            if (q.lanes == 32) return store ? launch_acc<NR, SGM_PF, true, true, 32>(ctx, q, nm) : launch_acc<NR, SGM_PF, true, false, 32>(ctx, q, nm);
            if (q.lanes == 24) return store ? launch_acc<NR, SGM_PF, false, true, 24>(ctx, q, nm) : launch_acc<NR, SGM_PF, false, false, 24>(ctx, q, nm);
        }
    }
    if (store) return full ? launch_acc<NR, SGM_PF, true, true, 0>(ctx, q, nm) : launch_acc<NR, SGM_PF, false, true, 0>(ctx, q, nm);
    return full ? launch_acc<NR, SGM_PF, true, false, 0>(ctx, q, nm) : launch_acc<NR, SGM_PF, false, false, 0>(ctx, q, nm);
}

static int launch_dirs(sva_ctx* ctx, const SgmParams& q, int nr, bool store) {
    switch (nr) {
        case 1: return launch_dirs_nr<1>(ctx, q, store);
        case 2: return launch_dirs_nr<2>(ctx, q, store);
        default: return launch_dirs_nr<4>(ctx, q, store);
    }
}

// smallest n in {2,4,8} disparities per lane with D % n == 0 and D / n <= 32
int sva_sgm_regs_per_lane(int D) {
    for (int n = 2; n <= 8; n *= 2)
        if (D % n == 0 && D / n <= 32) return n / 2;
    return 0;
}

// direction indices in the oracle's ORC_DIRS order: 0 v+, 1 v-, 2 h+, 3 h-, 4..7 diagonals
static const int DIRS[8][2] = {{0, 1}, {0, -1}, {1, 0}, {-1, 0}, {1, 1}, {-1, 1}, {1, -1}, {-1, -1}};

static void set_dirs(SgmParams& q, const int* idx, int n) {
    q.ndirs = n;
    for (int i = 0; i < n; i++) { q.dxs[i] = DIRS[idx[i]][0]; q.dys[i] = DIRS[idx[i]][1]; }
}

// One group of directions that sweep the rows the same way.  They share a row's C and S lines in L2 only while ALL their lines are
// resident and paced; a group with more lines than fit one resident wave (3 x 3840 at c3) is therefore cut into launches that do fit
// instead of running in unsynchronised waves that share nothing.  Such a group is always a ROW BLOCK (a whole frame that needs the cut is
// marched in row blocks: run_group_in_blocks), and it is cut by COLUMNS.
static int launch_row_group(sva_ctx* ctx, SgmParams& q, int nr, const int* idx, int n) {
    set_dirs(q, idx, n);
    q.ranged = 0;
    const int cap = sgm_resident_lines(ctx, nr);
    if (!sgm_paced(ctx, q) || n * q.W <= cap || q.W > cap) return launch_dirs(ctx, q, nr, false);
    // Launch j takes, of every direction, the lines that enter the block inside column range j.  A diagonal drifts one column per row, so
    // over a block of B rows the lines of a launch stay within their column range + B columns: each launch streams ITS columns of C and S
    // once for all three directions, and only the B-column fringe is streamed by two launches — (1 + B / range) volumes of traffic per group
    // instead of one per launch (c3, 270-row blocks: 1.14 instead of 2).
    const int W = q.W, launches = div_up(n * W, cap);
    const long long t = q.dys[0] > 0 ? q.row_y0 : q.H - 1 - (q.row_y0 + q.row_cnt - 1);  // rows the sweep has crossed before this block
    for (int j = 0; j < launches; j++) {
        const int c0 = (int)((long long)W * j / launches), c1 = (int)((long long)W * (j + 1) / launches);
        SgmParams s = q;
        s.ranged = 1; s.ndirs = 0;
        for (int dir = 0; dir < n; dir++) {
            // column of line x0 after t rows is (x0 + dx * t) mod W, so the lines entering in [c0, c1) are the range starting at (c0 - dx * t) mod W
            const int lo = (int)((((long long)c0 - (long long)q.dxs[dir] * t) % W + W) % W), len = c1 - c0, first = std::min(len, W - lo);
            for (int part = 0; part < 2; part++) {
                const int a = part == 0 ? lo : 0, cnt = part == 0 ? first : len - first;
                if (cnt <= 0) continue;
                s.dxs[s.ndirs] = q.dxs[dir]; s.dys[s.ndirs] = q.dys[dir]; s.state_slot[s.ndirs] = q.state_slot[dir];
                s.line_lo[s.ndirs] = a; s.line_cnt[s.ndirs] = cnt; s.ndirs++;
            }
        }
        SVA_TRY(launch_dirs(ctx, s, nr, false));
    }
    return SVA_OK;
}

// A row-sweeping group of a WHOLE frame that does not fit one resident wave (3 x 3840 lines at c3): the frame is marched in row blocks of
// about W / 16 rows — the row-block pipeline of the multi-GPU scheme on one GPU, the path-line state handed from block to block through two
// small buffers — because a block can be cut by columns (launch_row_group above), which a whole frame cannot (its diagonals cross every column).
static int run_group_in_blocks(sva_ctx* ctx, SgmParams& q, int nr, const int* idx, int n) {
    const int W = q.W, H = q.H, D = q.D;
    const int B = std::min(H, std::max(64, W / 16));
    const int blocks = div_up(H, B);
    const size_t state = (((size_t)3 * W * D * sizeof(uint16_t)) + 255) & ~(size_t)255;
    SVA_TRY(ctx->reserve(ctx->sgm_state, 2 * state));
    uint16_t* buf[2] = {ctx->sgm_state.as<uint16_t>(), (uint16_t*)(ctx->sgm_state.as<uint8_t>() + state)};
    const bool down = DIRS[idx[0]][1] > 0;
    for (int b = 0; b < blocks; b++) {
        const int blk = down ? b : blocks - 1 - b;  // in sweep order
        SgmParams s = q;
        s.row_y0 = blk * B; s.row_cnt = std::min(H, s.row_y0 + B) - s.row_y0;
        s.state_in = b > 0 ? buf[(b + 1) & 1] : nullptr;
        s.state_out = b + 1 < blocks ? buf[b & 1] : nullptr;
        for (int i = 0; i < 3; i++) s.state_slot[i] = i;
        SVA_TRY(launch_row_group(ctx, s, nr, idx, n));
    }
    return SVA_OK;
}

static bool group_needs_blocks(sva_ctx* ctx, const SgmParams& q, int nr, int n) {
    const int cap = sgm_resident_lines(ctx, nr);
    return sgm_paced(ctx, q) && n * q.W > cap && q.W <= cap && q.c_ds == 0;
}

// exactly the directions of dir_mask, one launch each: the first stores, the others RED, so S ends up as their sum
static int run_dir_mask(sva_ctx* ctx, SgmParams& q, int nr, uint32_t dir_mask) {
    bool first = true;
    for (int i = 0; i < 8; i++) {
        if (!(dir_mask & (1u << i))) continue;
        set_dirs(q, &i, 1);
        SVA_TRY(launch_dirs(ctx, q, nr, first));
        first = false;
    }
    return SVA_OK;
}

static int fill_params(sva_ctx* ctx, SgmParams& q, const uint16_t* C, int c_ds) {
    const sva_params& p = ctx->prm;
    const int nr = sva_sgm_regs_per_lane(p.num_disp);
    q.C = C; q.S = ctx->S.as<uint16_t>(); q.W = p.width; q.H = p.height; q.D = p.num_disp; q.c_ds = c_ds;
    q.p1p1 = (uint32_t)p.p1 * 0x10001u; q.p2p2 = (uint32_t)p.p2 * 0x10001u;
    q.lanes = nr ? p.num_disp / (2 * nr) : 0;
    q.elem_bytes = 2;
    return nr;
}

// Selected path directions on an EXTERNAL cost volume, optionally slice-major (multi-GPU: every rank gathers all disparity slices and
// aggregates its share of the directions; the partial sums are then reduce-scattered by rows).  ctx->S ends up as the sum of exactly
// these directions.  bit i = direction i of {v+, v-, h+, h-, d++, d-+, d+-, d--}.
int sva_run_sgm_dirs(sva_ctx* ctx, const uint16_t* Cext, int c_ds, uint32_t dir_mask, int rows_alloc) {
    const sva_params& p = ctx->prm;
    const int W = p.width, H = p.height, D = p.num_disp;
    const int nr = sva_sgm_regs_per_lane(D);
    if (nr == 0) return ctx->fail(SVA_ERR_BAD_ARG, "unsupported num_disp");
    if (c_ds > 0 && (D % c_ds || c_ds % (2 * nr))) return ctx->fail(SVA_ERR_BAD_ARG, "slice size must divide num_disp and hold whole lanes");
    if (!(dir_mask & 0xFFu)) return ctx->fail(SVA_ERR_BAD_ARG, "empty direction mask");
    if (rows_alloc < H) rows_alloc = H;
    if ((double)W * rows_alloc * D >= 4294967296.0) return ctx->fail(SVA_ERR_BAD_ARG, "padded volume too large for 32-bit element cursors");
    SVA_TRY(ctx->reserve(ctx->S, (size_t)W * rows_alloc * D * sizeof(uint16_t) + 64));
    if (rows_alloc > H)  // padding rows (the reduce-scatter wants equal row blocks) must read as zero
        SVA_CUDA_OK(ctx, cudaMemsetAsync(ctx->S.as<uint16_t>() + (size_t)W * H * D, 0, (size_t)W * (rows_alloc - H) * D * sizeof(uint16_t), ctx->stream));
    SgmParams q{};
    fill_params(ctx, q, Cext, c_ds);
    SVA_TRY(run_dir_mask(ctx, q, nr, dir_mask & 0xFFu));
    ctx->have_sgm = true;
    return SVA_OK;
}

// One direction group of the frame on image rows [y0, y0 + rows) only, accumulated (RED) into those rows of ctx->S, which the caller has
// zeroed: group 0 = {v+, d++, d-+} (sweeps down), 1 = {v-, d+-, d--} (sweeps up), 2 = {h+, h-}.  state_in / state_out: [3][W][D] u16 device
// buffers carrying L of every path line across the block boundary (nullptr at the sweep's first / last block); unused for group 2.
int sva_run_sgm_rows(sva_ctx* ctx, int group, int y0, int rows, const uint16_t* state_in, uint16_t* state_out) {
    const sva_params& p = ctx->prm;
    const int W = p.width, H = p.height, D = p.num_disp;
    const int nr = sva_sgm_regs_per_lane(D);
    if (nr == 0) return ctx->fail(SVA_ERR_BAD_ARG, "unsupported num_disp");
    if (group < 0 || group > 2 || y0 < 0 || rows < 1 || y0 + rows > H) return ctx->fail(SVA_ERR_BAD_ARG, "sgm_rows: bad group or row block");
    if (p.n_paths != 8) return ctx->fail(SVA_ERR_BAD_ARG, "sgm_rows: 8 paths only");
    if (!ctx->S.p || ctx->S.bytes < (size_t)W * H * D * sizeof(uint16_t)) return ctx->fail(SVA_ERR_STATE, "sgm_rows: no aggregation volume (sva_frame_rows_begin first)");
    SgmParams q{};
    fill_params(ctx, q, ctx->C.as<uint16_t>(), 0);
    static const int grp[3][3] = {{0, 4, 5}, {1, 6, 7}, {2, 3, -1}};
    if (group == 2) {  // the rows are the lines: a ranged launch of the ordinary march
        set_dirs(q, grp[2], 2);
        q.ranged = 1;
        for (int i = 0; i < 2; i++) { q.line_lo[i] = y0; q.line_cnt[i] = rows; }
        return launch_dirs(ctx, q, nr, false);
    }
    const bool first_block = group == 0 ? y0 == 0 : y0 + rows == H, last_block = group == 0 ? y0 + rows == H : y0 == 0;
    if (!first_block && !state_in) return ctx->fail(SVA_ERR_BAD_ARG, "sgm_rows: this block continues a sweep and needs state_in");
    q.row_y0 = y0; q.row_cnt = rows;
    q.state_in = first_block ? nullptr : state_in;
    q.state_out = last_block ? nullptr : state_out;
    for (int i = 0; i < 3; i++) q.state_slot[i] = i;
    return launch_row_group(ctx, q, nr, grp[group], 3);
}

int sva_run_sgm(sva_ctx* ctx) {
    const sva_params& p = ctx->prm;
    const int W = p.width, H = p.height, D = p.num_disp, n = p.n_paths;
    const int nr = sva_sgm_regs_per_lane(D);
    if (nr == 0) return ctx->fail(SVA_ERR_BAD_ARG, "num_disp must be a multiple of 2 with D/8 <= 32 (8..256)");
    const size_t cells = (size_t)W * H * D;
    SVA_TRY(ctx->reserve(ctx->S, cells * sizeof(uint16_t) + 64));
    SVA_TRY(ctx->reserve(ctx->disp, (size_t)W * H * sizeof(uint16_t)));
    SVA_TRY(ctx->reserve(ctx->subpix, (size_t)W * H * sizeof(float)));
    SgmParams q{};
    fill_params(ctx, q, ctx->C.as<uint16_t>(), 0);
    if (ctx->sgm_dir_mask_override) {  // test hook: S = the sum of exactly these directions, no K3
        SVA_TRY(run_dir_mask(ctx, q, nr, ctx->sgm_dir_mask_override));
        ctx->have_sgm = true;
        return SVA_OK;
    }
    if (n == 0) {  // no aggregation: K3 straight on the cost volume
        SVA_TRY(sva_run_wta(ctx, ctx->C.as<uint16_t>()));
        ctx->have_sgm = false; ctx->have_disp = true;
        return SVA_OK;
    }
    // wall time of the aggregation stage (its launches may overlap: entry "stage:k2_sgm" of the timing table, not a kernel)
    struct StageWall {
        sva_ctx* c; cudaEvent_t beg = nullptr, end = nullptr;
        explicit StageWall(sva_ctx* ctx) : c(ctx) {
            if (!c->timing) return;
            while (c->event_pool.size() < c->events_used + 2) { cudaEvent_t e; cudaEventCreate(&e); c->event_pool.push_back(e); }
            beg = c->event_pool[c->events_used]; end = c->event_pool[c->events_used + 1];
            c->events_used += 2;
            cudaEventRecord(beg, c->stream);
        }
        void stop() {
            if (!beg) return;
            cudaEventRecord(end, c->stream);
            c->ktimes.push_back(KernelTime{"stage:k2_sgm", beg, end});
            beg = nullptr;
        }
    } wall(ctx);
    if (n == 8) {
        // A row-sweeping launch holds only lines that advance one row per step, so (paced where a row is large) all of them touch a
        // row's C and S lines while these are in L2.  The horizontal lines (W steps each, every row in flight at once) cannot share
        // and get launches of their own.  S is never zeroed: the first horizontal direction WRITES it (plain stores: C in, S out = 4 B/DE),
        // the second accumulates (6 B/DE), then the row-sweeping groups — 10 B/DE for the horizontal pair instead of 12 plus the 2 B/DE of a memset
        static const int grp[2][3] = {{0, 4, 5}, {1, 6, 7}};
        const int h0 = 2, h1 = 3;
        set_dirs(q, &h0, 1);
        SVA_TRY(launch_dirs(ctx, q, nr, true));
        // The second horizontal direction is a launch of H warps bound by the latency of its own recurrence (~200 clocks per step): with
        // SVA_SGM_HSTORE = 2 (the default) it runs on the second stream NEXT TO the first row-sweeping group (REDs commute; both start after
        // the stores); 1 keeps the launches one after the other.
        const bool side = ctx->tune_sgm_hstore == 2 && q.W * (size_t)q.D * 4 < 768 * 1024;  // not next to paced launches: they want the SM to themselves
        cudaStream_t main_stream = ctx->stream;
        if (side) {
            if (!ctx->aux_stream) {
                SVA_CUDA_OK(ctx, cudaStreamCreateWithFlags(&ctx->aux_stream, cudaStreamNonBlocking));
                SVA_CUDA_OK(ctx, cudaEventCreateWithFlags(&ctx->ev_fork, cudaEventDisableTiming));
            }
            if (!ctx->ev_zero) SVA_CUDA_OK(ctx, cudaEventCreateWithFlags(&ctx->ev_zero, cudaEventDisableTiming));
            SVA_CUDA_OK(ctx, cudaEventRecord(ctx->ev_fork, main_stream));
            SVA_CUDA_OK(ctx, cudaStreamWaitEvent(ctx->aux_stream, ctx->ev_fork, 0));
            ctx->stream = ctx->aux_stream;
        }
        set_dirs(q, &h1, 1);
        const int rc_h1 = launch_dirs(ctx, q, nr, false);
        if (side) {
            ctx->stream = main_stream;
            if (rc_h1 == SVA_OK) SVA_CUDA_OK(ctx, cudaEventRecord(ctx->ev_zero, ctx->aux_stream));
        }
        SVA_TRY(rc_h1);
        for (int g = 0; g < 2; g++) {
            if (group_needs_blocks(ctx, q, nr, 3)) SVA_TRY(run_group_in_blocks(ctx, q, nr, grp[g], 3));
            else SVA_TRY(launch_row_group(ctx, q, nr, grp[g], 3));
        }
        if (side) SVA_CUDA_OK(ctx, cudaStreamWaitEvent(main_stream, ctx->ev_zero, 0));
        wall.stop();
        SVA_TRY(sva_run_wta(ctx, ctx->S.as<uint16_t>()));
        ctx->have_sgm = true; ctx->have_disp = true;
        return SVA_OK;
    }
    // 4 paths: S = 0 (zeroed next to K1a / K1b when the caller got that far ahead: sva_api.cu), one launch accumulating with REDs, K3 reads S_total
    if (ctx->s_prezeroed) SVA_CUDA_OK(ctx, cudaStreamWaitEvent(ctx->stream, ctx->ev_zero, 0));
    else SVA_CUDA_OK(ctx, cudaMemsetAsync(ctx->S.p, 0, cells * sizeof(uint16_t), ctx->stream));
    ctx->s_prezeroed = false;
    static const int all4[4] = {0, 1, 2, 3};
    set_dirs(q, all4, 4);
    SVA_TRY(launch_dirs(ctx, q, nr, false));
    wall.stop();
    SVA_TRY(sva_run_wta(ctx, ctx->S.as<uint16_t>()));
    ctx->have_sgm = true; ctx->have_disp = true;
    return SVA_OK;
}
