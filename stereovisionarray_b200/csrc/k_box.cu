// k_box.cu — K1b: 2k x 2k box sum of the AD volume + shift/cap packing + cell validity.
//
//   C_raw(y,x,d) = sum_{j,i in [-k,k)} A(y+j, x+i, d)            (half-open window — reference src/CameraStereoVision.cpp:57,77)
//   PACK_U16: C = valid ? min(cap, C_raw >> shift) : cap           RAW_U32: C = valid ? C_raw : 0xFFFFFFFF
//
// Two kernels: k_box_planar (below, the volume pipeline's hot path, reads the planar AD volume) and the general k_box_cost
// ([H][W][D] u16 in, PACK_U16 or RAW_U32 out; literal mode, improveWithDisparity and the RAW recomputation use it):
// A CTA of k_box_cost owns a strip of TXi = 16*NC columns x 32 disparities and marches down a band of rows.  Each thread keeps the
// vertical running sums V of NC consecutive columns x 2 disparities in registers (add the row entering the window,
// subtract the row leaving it).  The horizontal window sum is a difference of row prefix sums: every thread scans its
// own NC columns in registers, segment totals are exchanged through shared memory, and the prefix row P lives in
// shared memory for the two look-ups P[x+k-1] - P[x-k-1].  All sums are exact u32.
#include <algorithm>

#include "sva_common.cuh"

#define BOX_THREADS 256
#define BOX_DP 16       // d-pairs per CTA  (32 disparities)
#define BOX_CG 16       // column groups per CTA
#define BOX_MAX_BAND 512

struct BoxParams {
    const uint16_t* A;
    void* out;
    int W, H, D, k, dmin, shift, cap;
    int gxp, gxn, gyp, gyn;  // largest positive / negative |offset| over all pairs, per axis (0 = none)
    int band_rows, txo;
    int apply_validity;
};

__device__ __forceinline__ int axis_limit(int pos, int dim, int k, int gp, int gn) {
    // largest delta >= 0 such that k <= pos - g*delta <= dim-k for every pair offset g on this axis; -1 if the pixel itself is outside [k, dim-k)
    if (pos < k || pos >= dim - k) return -1;
    int lim = 0x7FFFFFFF;
    if (gp > 0) lim = min(lim, (pos - k) / gp);
    if (gn > 0) lim = min(lim, (dim - k - pos) / gn);
    return lim;
}

#define BOX_STAGES 3

// 16-byte async copy global -> shared; src_bytes == 0 zero-fills (out-of-image rows / columns / disparities)
__device__ __forceinline__ void box_cp16(uint32_t dst, const void* src, int src_bytes) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(src_bytes) : "memory");
}

template <int NC, bool RAW>
__global__ void __launch_bounds__(BOX_THREADS, NC == 8 ? 3 : 4)
k_box_cost(BoxParams q) {
    constexpr int TXI = BOX_CG * NC;
    constexpr int ROW_BYTES = TXI * 64;                 // one tile row: TXI columns x 32 disparities x u16
    constexpr int STAGE_BYTES = 2 * ROW_BYTES;          // [entering row][leaving row]
    extern __shared__ __align__(16) unsigned char box_smem[];
    unsigned char* s_ring = box_smem;                                         // BOX_STAGES * STAGE_BYTES
    uint2 (*s_P)[BOX_DP] = reinterpret_cast<uint2 (*)[BOX_DP]>(box_smem + BOX_STAGES * STAGE_BYTES);      // [TXI][BOX_DP]
    uint2 (*s_tot)[BOX_DP] = reinterpret_cast<uint2 (*)[BOX_DP]>(box_smem + BOX_STAGES * STAGE_BYTES + TXI * BOX_DP * 8);  // [BOX_CG][BOX_DP]
    int* s_limy = reinterpret_cast<int*>(box_smem + BOX_STAGES * STAGE_BYTES + TXI * BOX_DP * 8 + BOX_CG * BOX_DP * 8);

    const int t = threadIdx.x, dp = t & (BOX_DP - 1), cg = t >> 4;
    const int W = q.W, H = q.H, D = q.D, k = q.k;
    const int d0 = blockIdx.y * 32;
    const int d = d0 + 2 * dp;
    const bool d_ok = d < D;
    const int xs = blockIdx.x * q.txo - k;  // global x of strip column 0
    const int y0 = blockIdx.z * q.band_rows, y1 = min(H, y0 + q.band_rows);
    if (y0 >= H) return;

    for (int i = t; i < y1 - y0; i += BOX_THREADS) s_limy[i] = q.apply_validity ? axis_limit(y0 + i, H, k, q.gyp, q.gyn) : 0x7FFFFFFF;

    int limx[NC];
    uint32_t v0[NC], v1[NC];
#pragma unroll
    for (int j = 0; j < NC; j++) {
        int x = xs + cg * NC + j;
        limx[j] = q.apply_validity ? axis_limit(x, W, k, q.gxp, q.gxn) : 0x7FFFFFFF;
        v0[j] = 0; v1[j] = 0;
    }
    const long long rowstride = (long long)W * D;
    const uint32_t ring_base = (uint32_t)__cvta_generic_to_shared(s_ring);

    // cooperative stage fill: the tile row is TXI * 4 chunks of 16 B (8 disparities); thread t copies chunks t, t + 256, ...
    auto fill = [&](int it) {  // iteration it: entering row y0 + it + k - 1, leaving row y0 + it - k (only once it >= 0)
        const uint32_t st = ring_base + ((it + 2 * k) % BOX_STAGES) * STAGE_BYTES;
        const int ra = y0 + it + k - 1, rs = y0 + it - k;
        const bool ra_ok = ra >= 0 && ra < H, rs_ok = it >= 0 && rs >= 0 && rs < H;
#pragma unroll
        for (int c = t; c < TXI * 4; c += BOX_THREADS) {
            const int col = c >> 2, part = c & 3, x = xs + col, dd = d0 + 8 * part;
            const bool in = x >= 0 && x < W && dd < D;
            const long long off = ((long long)(in ? x : 0)) * D + (in ? dd : 0);
            box_cp16(st + c * 16, q.A + (ra_ok ? ra : 0) * rowstride + off, (in && ra_ok) ? 16 : 0);
            if (it >= 0) box_cp16(st + ROW_BYTES + c * 16, q.A + (rs_ok ? rs : 0) * rowstride + off, (in && rs_ok) ? 16 : 0);
        }
    };

    const int it_begin = -(2 * k - 1), it_end = y1 - y0;  // warm-up iterations (it < 0) only accumulate
#pragma unroll
    for (int i = 0; i < BOX_STAGES - 1; i++) {
        if (it_begin + i < it_end) fill(it_begin + i);
        asm volatile("cp.async.commit_group;" ::: "memory");
    }

    for (int it = it_begin; it < it_end; it++) {
        asm volatile("cp.async.wait_group %0;" ::"n"(BOX_STAGES - 2) : "memory");
        __syncthreads();  // stage `it` is complete for every thread; everyone has finished reading stage it-1
        if (it + BOX_STAGES - 1 < it_end) fill(it + BOX_STAGES - 1);
        asm volatile("cp.async.commit_group;" ::: "memory");
        const unsigned char* st = s_ring + ((it + 2 * k) % BOX_STAGES) * STAGE_BYTES;
        const uint32_t* rowa = reinterpret_cast<const uint32_t*>(st) + (cg * NC) * 16 + dp;  // [col][16 u32]
#pragma unroll
        for (int j = 0; j < NC; j++) { uint32_t w = rowa[j * 16]; v0[j] += w & 0xFFFFu; v1[j] += w >> 16; }
        if (it < 0) continue;
        const int y = y0 + it;
        // prefix over this thread's columns
        uint32_t p0[NC], p1[NC];
        uint32_t a0 = 0, a1 = 0;
#pragma unroll
        for (int j = 0; j < NC; j++) { a0 += v0[j]; a1 += v1[j]; p0[j] = a0; p1[j] = a1; }
        s_tot[cg][dp] = make_uint2(a0, a1);
        __syncthreads();
        uint32_t o0 = 0, o1 = 0;
        for (int g = 0; g < cg; g++) { uint2 tt = s_tot[g][dp]; o0 += tt.x; o1 += tt.y; }
#pragma unroll
        for (int j = 0; j < NC; j++) s_P[cg * NC + j][dp] = make_uint2(p0[j] + o0, p1[j] + o1);
        __syncthreads();
        const int limy = s_limy[it];
#pragma unroll
        for (int j = 0; j < NC; j++) {
            int ci = cg * NC + j, x = xs + ci;
            if (ci < k || ci > TXI - k || x >= W || ci - k >= q.txo || !d_ok) continue;
            uint2 hi = s_P[ci + k - 1][dp];
            uint2 lo = (ci - k - 1 >= 0) ? s_P[ci - k - 1][dp] : make_uint2(0u, 0u);
            uint32_t r0 = hi.x - lo.x, r1 = hi.y - lo.y;
            int lim = min(limx[j], limy);
            bool ok0 = q.dmin + d <= lim, ok1 = q.dmin + d + 1 <= lim;
            long long o = ((long long)y * W + x) * D + d;
            if (RAW) {
                *reinterpret_cast<uint2*>((uint32_t*)q.out + o) = make_uint2(ok0 ? r0 : 0xFFFFFFFFu, ok1 ? r1 : 0xFFFFFFFFu);
            } else {
                uint32_t c0 = ok0 ? min((uint32_t)q.cap, r0 >> q.shift) : (uint32_t)q.cap;
                uint32_t c1 = ok1 ? min((uint32_t)q.cap, r1 >> q.shift) : (uint32_t)q.cap;
                *reinterpret_cast<uint32_t*>((uint16_t*)q.out + o) = c0 | (c1 << 16);
            }
        }
        const uint32_t* rows = reinterpret_cast<const uint32_t*>(st + ROW_BYTES) + (cg * NC) * 16 + dp;
#pragma unroll
        for (int j = 0; j < NC; j++) { uint32_t w = rows[j * 16]; v0[j] -= w & 0xFFFFu; v1[j] -= w >> 16; }
    }
}

template <int NC, bool RAW>
static cudaError_t box_launch(const BoxParams& q, dim3 grid, cudaStream_t stream) {
    constexpr int TXI = BOX_CG * NC;
    const size_t smem = (size_t)BOX_STAGES * 2 * TXI * 64 + (size_t)TXI * BOX_DP * 8 + BOX_CG * BOX_DP * 8 + BOX_MAX_BAND * 4;
    cudaError_t e = cudaFuncSetAttribute(k_box_cost<NC, RAW>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    k_box_cost<NC, RAW><<<grid, BOX_THREADS, smem, stream>>>(q);
    return cudaGetLastError();
}

// A -> out (u16 packed or u32 raw).  D must be a multiple of 8 (16-byte async copies).  Used by the volume pipeline and (raw, no validity) by literal mode / refine.
int sva_launch_box(sva_ctx* ctx, const uint16_t* A, void* out, int W, int H, int D, int k, const sva_params* prm, bool raw, bool apply_validity) {
    if (k < 1 || k > 56) return ctx->fail(SVA_ERR_BAD_ARG, "win_half must be in 1..56");
    if (D % 8) return ctx->fail(SVA_ERR_BAD_ARG, "box filter needs a multiple of 8 planes");
    BoxParams q{};
    q.A = A; q.out = out; q.W = W; q.H = H; q.D = D; q.k = k;
    q.dmin = prm ? prm->min_disp : 0; q.shift = prm ? prm->cost_shift : 0; q.cap = prm ? prm->cost_cap : SVA_COST_CAP_MAX;
    q.apply_validity = apply_validity ? 1 : 0;
    if (prm && apply_validity) {
        for (int i = 0; i < prm->n_pairs; i++) {
            int gx = prm->pair_gx[i], gy = prm->pair_gy[i];
            if (gx > 0) q.gxp = gx > q.gxp ? gx : q.gxp;
            if (gx < 0) q.gxn = -gx > q.gxn ? -gx : q.gxn;
            if (gy > 0) q.gyp = gy > q.gyp ? gy : q.gyp;
            if (gy < 0) q.gyn = -gy > q.gyn ? -gy : q.gyn;
        }
    }
    const bool wide = k > 12;
    const int txi = wide ? 128 : 64;
    q.txo = txi - 2 * k + 1;
    int strips = div_up(W, q.txo), dch = div_up(D, 32);
    // enough CTAs for one full wave, bands no shorter than 4k rows (warm-up is 2k-1 rows of loads)
    int bands = div_up(2 * ctx->sm_count * 2, strips * dch);
    int min_band = 4 * k > 32 ? 4 * k : 32;
    if (bands > H / min_band) bands = H / min_band;
    if (bands < 1) bands = 1;
    if (div_up(H, bands) > BOX_MAX_BAND) bands = div_up(H, BOX_MAX_BAND);
    q.band_rows = div_up(H, bands);
    bands = div_up(H, q.band_rows);
    dim3 grid(strips, dch, bands);
    LaunchScope ls(ctx, raw ? "k_box_cost_raw" : "k_box_cost");
    cudaError_t e;
    if (wide) e = raw ? box_launch<8, true>(q, grid, ctx->stream) : box_launch<8, false>(q, grid, ctx->stream);
    else e = raw ? box_launch<4, true>(q, grid, ctx->stream) : box_launch<4, false>(q, grid, ctx->stream);
    SVA_CUDA_OK(ctx, e);
    return SVA_OK;
}

// ---- K1b on the planar AD volume (the volume pipeline's hot path) -------------------------------------------------------------
// A warp owns ONE disparity pair (a u16x2 word per pixel) of a 256-column strip and marches down a band of rows; a lane owns 8
// consecutive columns, i.e. 32 contiguous bytes of a plane row: two 16-byte streaming loads for the row entering the window and
// two for the row leaving it, straight from global memory (zero borders in the layout: no bounds checks, no staging).
//   vertical:   u = enter - leave + 0x80008000 keeps both u16 fields positive, so ONE subtraction updates two cells:
//               F += u (the whole word, fields bleed on purpose) and Vh += u >> 16 (odd cell).  Sums are linear, so the even
//               cell is recovered after the horizontal sum as dF - (dVh << 16); the per-row bias is a constant (arithmetic mod 2^32).
//   horizontal: in-register prefix over the lane's 8 columns, warp shuffle scan of the lane totals, then the window sum is
//               T[c + k] - T[c - k] on a per-warp table in shared memory (stored by (index mod 8) rows: conflict-free).
// No __syncthreads in the arithmetic: the 8 warps of a CTA (8 d-pairs = 16 disparities = one 32-byte sector per pixel) only
// meet to transpose their packed results through shared memory into 16-byte coalesced stores of C [H][W][D].
#define BXP_WARPS 8
#define BXP_TCOLS 48    // table row: 8 guard columns + 33 + 7 guard columns
#define BXP_OPITCH 260  // words per staged output row (== 4 mod 32: the two halves of a pixel fall into different banks)
#define BXP_MAX_BAND 1024

struct BoxPParams {
    const uint32_t* AP;
    uint16_t* C;
    int W, H, D, k, kk, dmin, shift, cap;
    int gxp, gxn, gyp, gyn;
    int band_rows, txo, wp;
    int chunk;  // k_box_planar_shfl: warm-up rows summed per horizontal pass (chunk x the largest A keeps a 16-bit field below 32768)
    long long row_words;
    int ry0, ry1;  // output rows [ry0, ry1) (the whole image, or a row block)
};

__global__ void __launch_bounds__(256, 2)
k_box_planar(BoxPParams q) {
    __shared__ __align__(16) uint32_t s_out[2][BXP_WARPS][BXP_OPITCH];
    __shared__ __align__(8) unsigned long long s_bar[2];  // one mbarrier per staging buffer: "all 8 warps have written this row's words"
    __shared__ uint2 s_T[BXP_WARPS][8 * BXP_TCOLS];
    __shared__ int s_limy[BXP_MAX_BAND];
    const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
    const int W = q.W, H = q.H, D = q.D, k = q.k;
    const int dpc = min((int)blockIdx.y * BXP_WARPS + warp, (D >> 1) - 1);  // warps beyond D/2 (D % 16 != 0) redo the last pair; never stored
    const int d = 2 * dpc;
    const int xs = blockIdx.x * q.txo - q.kk;  // image x of strip column 0
    const int y0 = q.ry0 + blockIdx.z * q.band_rows, y1 = min(q.ry1, y0 + q.band_rows);
    for (int i = t; i < y1 - y0; i += 256) s_limy[i] = axis_limit(y0 + i, H, k, q.gyp, q.gyn);

    int thr[8], thrmin = 0x7FFFFFFF;  // validity slack of each column for this warp's even disparity
#pragma unroll
    for (int j = 0; j < 8; j++) {
        thr[j] = axis_limit(xs + lane * 8 + j, W, k, q.gxp, q.gxn) - q.dmin - d;
        thrmin = min(thrmin, thr[j]);
    }
    uint2* tbl = &s_T[warp][8 + lane];
    if (lane == 0) tbl[0] = make_uint2(0u, 0u);  // T[0] = 0 (never overwritten)
    const uint32_t bar0 = (uint32_t)__cvta_generic_to_shared(&s_bar[0]);
    if (t == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar0), "r"(BXP_WARPS) : "memory");
        asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar0 + 8), "r"(BXP_WARPS) : "memory");
    }
    int offh[8], offl[8];
#pragma unroll
    for (int j = 0; j < 8; j++) {
        offh[j] = ((j + k) & 7) * BXP_TCOLS + ((j + k) >> 3);
        offl[j] = ((j - k) & 7) * BXP_TCOLS + ((j - k) >> 3);  // arithmetic shift: floor
    }
    __syncthreads();

    const uint32_t* pz = q.AP + (size_t)dpc * q.wp + (size_t)blockIdx.x * q.txo + lane * 8;  // physical row 0: zeros
    const uint32_t* pe = pz + (size_t)y0 * q.row_words;  // update n adds physical row y0 + n (image row y0 - k + n)
    const long long back = 2LL * k * q.row_words;
    const int N = (y1 - y0) + 2 * k - 1;
    uint32_t F[8], Vh[8];
#pragma unroll
    for (int j = 0; j < 8; j++) { F[j] = 0; Vh[j] = 0; }

    // per-thread output items: (column, half) pairs -> one 16-byte store each, pointers advance one image row per output row
    const int hf = t & 1;
    const bool half_ok = (int)blockIdx.y * 16 + 8 * hf < D;
    const int xl0 = t >> 1, xl1 = xl0 + 128;
    const bool st0 = half_ok && xl0 >= q.kk && xl0 < q.kk + q.txo && xs + xl0 < W;
    const bool st1 = half_ok && xl1 >= q.kk && xl1 < q.kk + q.txo && xs + xl1 < W;
    uint16_t* po = q.C + ((size_t)y0 * W + (xs + xl0)) * D + blockIdx.y * 16 + 8 * hf;  // item 1 is 128 columns further
    const size_t orow = (size_t)W * D;
    const uint32_t kB = (uint32_t)k << 16;

    // transposed store of output row r (all 8 warps' words of that row are in s_out[r & 1] once the barrier's phase r >> 1 has completed)
    auto store_row = [&](const int r) {
        const uint32_t bar = bar0 + 8 * (r & 1), parity = (uint32_t)(r >> 1) & 1u;
        asm volatile(
            "{\n"
            ".reg .pred p;\n"
            "BOXWAIT_%=:\n"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
            "@p bra BOXDONE_%=;\n"
            "bra BOXWAIT_%=;\n"
            "BOXDONE_%=:\n"
            "}" ::"r"(bar), "r"(parity) : "memory");
        const uint32_t* src = &s_out[r & 1][4 * hf][xl0];
        if (st0) *reinterpret_cast<uint4*>(po) = make_uint4(src[0], src[BXP_OPITCH], src[2 * BXP_OPITCH], src[3 * BXP_OPITCH]);
        if (st1) *reinterpret_cast<uint4*>(po + 128 * D) = make_uint4(src[128], src[BXP_OPITCH + 128], src[2 * BXP_OPITCH + 128], src[3 * BXP_OPITCH + 128]);
        po += orow;
    };
    // one update + (once the window is full) one output row; cur = this row's words, the caller keeps the next row's loads in flight
    auto row = [&](const int n, const uint4& e0, const uint4& e1, const uint4& l0, const uint4& l1) {
        {
            const uint32_t ee[8] = {e0.x, e0.y, e0.z, e0.w, e1.x, e1.y, e1.z, e1.w};
            const uint32_t ll[8] = {l0.x, l0.y, l0.z, l0.w, l1.x, l1.y, l1.z, l1.w};
#pragma unroll
            for (int j = 0; j < 8; j++) {
                const uint32_t u = ee[j] - ll[j] + 0x80008000u;
                F[j] += u;
                Vh[j] += u >> 16;
            }
        }
        if (n < 2 * k - 1) return;
        const int it = n - (2 * k - 1);
        uint32_t pF[8], pV[8];
        pF[0] = F[0]; pV[0] = Vh[0];
#pragma unroll
        for (int j = 1; j < 8; j++) { pF[j] = pF[j - 1] + F[j]; pV[j] = pV[j - 1] + Vh[j]; }
        uint32_t incF = pF[7], incV = pV[7];
#pragma unroll
        for (int s = 1; s < 32; s <<= 1) {
            const uint32_t a = __shfl_up_sync(0xffffffffu, incF, s), b = __shfl_up_sync(0xffffffffu, incV, s);
            if (lane >= s) { incF += a; incV += b; }
        }
        const uint32_t exF = incF - pF[7], exV = incV - pV[7];
        __syncwarp();
#pragma unroll
        for (int j = 0; j < 8; j++)  // T[c + 1] = inclusive prefix up to column c = lane*8 + j
            tbl[((j + 1) & 7) * BXP_TCOLS + ((j + 1) >> 3)] = make_uint2(pF[j] + exF, pV[j] + exV);
        __syncwarp();
        // bias of a 2k-column window after n + 1 updates: B on the odd cell, B * 65537 on the whole-word sum
        const uint32_t B = (uint32_t)(n + 1) * kB, B2 = B * 65537u;
        const int srow = s_limy[it] - q.dmin - d;
        uint32_t w[8];
        if (__all_sync(0xffffffffu, min(thrmin, srow) >= 1)) {  // every cell of the warp's 256 x 2 cells is valid (the image interior)
#pragma unroll
            for (int j = 0; j < 8; j++) {
                const uint2 hi = tbl[offh[j]], lo = tbl[offl[j]];
                const uint32_t chi = hi.y - lo.y - B;
                const uint32_t clo = hi.x - lo.x - B2 - (chi << 16);
                const uint32_t c0 = min(clo >> q.shift, (uint32_t)q.cap), c1 = min(chi >> q.shift, (uint32_t)q.cap);
                w[j] = c1 * 65536u + c0;
            }
        } else {
#pragma unroll
            for (int j = 0; j < 8; j++) {
                const uint2 hi = tbl[offh[j]], lo = tbl[offl[j]];
                const uint32_t chi = hi.y - lo.y - B;
                const uint32_t clo = hi.x - lo.x - B2 - (chi << 16);
                uint32_t c0 = min(clo >> q.shift, (uint32_t)q.cap), c1 = min(chi >> q.shift, (uint32_t)q.cap);
                const int m = min(thr[j], srow);
                c0 = m >= 0 ? c0 : (uint32_t)q.cap;
                c1 = m >= 1 ? c1 : (uint32_t)q.cap;
                w[j] = c1 * 65536u + c0;
            }
        }
        // The 8 warps meet through a SPLIT barrier instead of __syncthreads: a warp announces its words of row `it` (mbarrier arrive) and
        // goes on; the transposed store of a row happens one row later, when that row's barrier phase has completed — so a warp only
        // ever waits for the others' PREVIOUS row, and the warps of a CTA drift up to a row apart instead of marching in phase through
        // the same pipes.  WAR on the double buffer: whoever writes buffer b for row it + 2 has passed the wait for row it + 1, i.e.
        // every warp has arrived for row it + 1, which each does after its store pass of row it.
        if (it > 0) store_row(it - 1);
        uint32_t* so = &s_out[it & 1][warp][lane * 8];
        *reinterpret_cast<uint4*>(so) = make_uint4(w[0], w[1], w[2], w[3]);
        *reinterpret_cast<uint4*>(so + 4) = make_uint4(w[4], w[5], w[6], w[7]);
        __syncwarp();
        if (lane == 0) asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar0 + 8 * (it & 1)) : "memory");
    };

    // software pipeline, unrolled by two so the row buffers ping-pong without register moves
    uint4 a0 = ldg_stream_u128(pe), a1 = ldg_stream_u128(pe + 4), al0 = make_uint4(0, 0, 0, 0), al1 = al0;
    uint4 b0 = a0, b1 = a1, bl0 = al0, bl1 = al1;
    auto fetch = [&](const int n, uint4& e0, uint4& e1, uint4& l0, uint4& l1) {  // loads of update n
        if (n < N) {
            pe += q.row_words;
            const uint32_t* pl = n >= 2 * k ? pe - back : pz;
            e0 = ldg_stream_u128(pe); e1 = ldg_stream_u128(pe + 4);
            l0 = ldg_stream_u128(pl); l1 = ldg_stream_u128(pl + 4);
        }
    };
    for (int n = 0; n < N; n += 2) {
        fetch(n + 1, b0, b1, bl0, bl1);
        row(n, a0, a1, al0, al1);
        if (n + 1 >= N) break;
        fetch(n + 2, a0, a1, al0, al1);
        row(n + 1, b0, b1, bl0, bl1);
    }
    store_row(y1 - y0 - 1);  // the last row's deferred store
}

// ---- K1b with the horizontal window sums in registers (win_half = K, K % 8 == 4: the configurations' K = 20, and 4, 12, 28, ...) ------
// Same mapping as k_box_planar (warp = one disparity pair of a 256-column strip, lane = 8 consecutive columns), but the accumulators
// are the WINDOW sums themselves, not column sums, and the per-warp prefix table in shared memory is gone.  Per row, u = enter - leave
// + 0x80008000 is one word per column with two 16-bit fields (|enter - leave| <= 32 pairs x 255 keeps both fields positive), and what
// the row adds to the window sum of column c is the sum of u over [c - K, c + K).  Because K % 8 == 4, the window of a lane's column 4
// is exactly the lanes l - M .. l + M (M = (K - 4) / 8): lane totals, 2M shuffles.  From there the window slides one column at a time,
//     dW(c + 1) = dW(c) + u(c + K) - u(c - K),
// three steps up and four steps down, and the columns entering / leaving are whole packed words of other lanes: 14 shuffles per row
// move BOTH cells of a word.  The two cells are carried as in k_box_planar: F = the whole-word sums (fields bleed, mod 2^32) and
// Hh = the odd cell alone; (int)(u_a - u_b + 0x8000) >> 16 is the odd field's difference exactly, because the even field's
// difference stays within +-32767.  Per row and 8 columns x 2 cells: 14 + 4M shuffles instead of 8 STS.64 + 16 LDS.64 + 10 shuffles.
// Warm-up rows (the 2K - 1 rows before a band's first output) have nothing leaving, so they are summed as packed words first —
// `chunk` rows at a time, as many as keep a field below 32768 — and only every chunk goes through the horizontal pass.
// A lane's 32 bytes of a row arrive in ONE 256-bit load (LDG.E.256: 1 KB of whole sectors per warp-instruction; two 128-bit loads per lane
// touch every sector twice).  PF = rows the loads run ahead of the arithmetic (1; 2 measured no faster), OCC = CTAs per SM the kernel is
// compiled for (2: up to 128 registers; 3: 80 registers, no spills — chosen per launch by sva_launch_box_planar's cost model).
template <int K, int PF, int OCC>
__global__ void __launch_bounds__(256, OCC)
k_box_planar_shfl(BoxPParams q) {
    static_assert(K % 8 == 4 && K >= 4 && K <= 56, "window half-width must be 4 mod 8");
    constexpr int M = (K - 4) / 8;
    __shared__ __align__(16) uint32_t s_out[2][BXP_WARPS][BXP_OPITCH];
    __shared__ __align__(8) unsigned long long s_bar[2];  // one mbarrier per staging buffer: "all 8 warps have written this row's words"
    __shared__ int s_limy[BXP_MAX_BAND];
    const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
    const int W = q.W, H = q.H, D = q.D;
    const int dpc = min((int)blockIdx.y * BXP_WARPS + warp, (D >> 1) - 1);  // warps beyond D/2 (D % 16 != 0) redo the last pair; never stored
    const int d = 2 * dpc;
    const int xs = blockIdx.x * q.txo - K;  // image x of strip column 0 (the left zero border is K columns: K % 4 == 0)
    const int y0 = q.ry0 + blockIdx.z * q.band_rows, y1 = min(q.ry1, y0 + q.band_rows);
    for (int i = t; i < y1 - y0; i += 256) s_limy[i] = axis_limit(y0 + i, H, K, q.gyp, q.gyn);

    int thr[8], thrmin = 0x7FFFFFFF;  // validity slack of each column for this warp's even disparity
#pragma unroll
    for (int j = 0; j < 8; j++) {
        thr[j] = axis_limit(xs + lane * 8 + j, W, K, q.gxp, q.gxn) - q.dmin - d;
        thrmin = min(thrmin, thr[j]);
    }
    const uint32_t bar0 = (uint32_t)__cvta_generic_to_shared(&s_bar[0]);
    if (t == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar0), "r"(BXP_WARPS) : "memory");
        asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar0 + 8), "r"(BXP_WARPS) : "memory");
    }
    __syncthreads();

    // L2 policy of the loads of A and the stores of C: evict_normal (entering rows evict_last, leaving rows and C evict_first measured no
    // gain: DESIGN.md §4)
    const unsigned long long pol = l2_policy_evict_normal();
    const uint32_t* pe = q.AP + (size_t)dpc * q.wp + (size_t)blockIdx.x * q.txo + lane * 8 + (size_t)y0 * q.row_words;  // update n adds physical row y0 + n (image row y0 - K + n)
    const long long back = 2LL * K * q.row_words;
    const int N = (y1 - y0) + 2 * K - 1;
    uint32_t F[8], Hh[8];
#pragma unroll
    for (int j = 0; j < 8; j++) { F[j] = 0; Hh[j] = 0; }

    // per-thread output items: (column, half) pairs -> one 16-byte store each, pointers advance one image row per output row
    const int hf = t & 1;
    const bool half_ok = (int)blockIdx.y * 16 + 8 * hf < D;
    const int xl0 = t >> 1, xl1 = xl0 + 128;
    const bool st0 = half_ok && xl0 >= K && xl0 < K + q.txo && xs + xl0 < W;
    const bool st1 = half_ok && xl1 >= K && xl1 < K + q.txo && xs + xl1 < W;
    uint16_t* po = q.C + ((size_t)y0 * W + (xs + xl0)) * D + blockIdx.y * 16 + 8 * hf;  // item 1 is 128 columns further
    const size_t orow = (size_t)W * D;

    // transposed store of output row r (all 8 warps' words of that row are in s_out[r & 1] once the barrier's phase r >> 1 has completed)
    auto store_row = [&](const int r) {
        const uint32_t bar = bar0 + 8 * (r & 1), parity = (uint32_t)(r >> 1) & 1u;
        asm volatile(
            "{\n"
            ".reg .pred p;\n"
            "BOXSWAIT_%=:\n"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
            "@p bra BOXSDONE_%=;\n"
            "bra BOXSWAIT_%=;\n"
            "BOXSDONE_%=:\n"
            "}" ::"r"(bar), "r"(parity) : "memory");
        const uint32_t* src = &s_out[r & 1][4 * hf][xl0];
        if (st0) stg_u128_hint(po, make_uint4(src[0], src[BXP_OPITCH], src[2 * BXP_OPITCH], src[3 * BXP_OPITCH]), pol);
        if (st1) stg_u128_hint(po + 128 * D, make_uint4(src[128], src[BXP_OPITCH + 128], src[2 * BXP_OPITCH + 128], src[3 * BXP_OPITCH + 128]), pol);
        po += orow;
    };
    // horizontal pass: the window sums of every column take in one row's (or one warm-up chunk's) packed differences u
    auto hpass = [&](const uint32_t (&u)[8]) {
        uint32_t tF = ((u[0] + u[1]) + (u[2] + u[3])) + ((u[4] + u[5]) + (u[6] + u[7]));
        uint32_t tH = (((u[0] >> 16) + (u[1] >> 16)) + ((u[2] >> 16) + (u[3] >> 16))) + (((u[4] >> 16) + (u[5] >> 16)) + ((u[6] >> 16) + (u[7] >> 16)));
        uint32_t dF[8], dH[8];
        dF[4] = tF; dH[4] = tH;
#pragma unroll
        for (int s = 1; s <= M; s++) {
            dF[4] += __shfl_up_sync(0xffffffffu, tF, s) + __shfl_down_sync(0xffffffffu, tF, s);
            dH[4] += __shfl_up_sync(0xffffffffu, tH, s) + __shfl_down_sync(0xffffffffu, tH, s);
        }
#pragma unroll
        for (int i = 0; i < 3; i++) {  // column 4 + i -> 5 + i: column 8(l + M + 1) + i enters, column 8(l - M) + i leaves
            const uint32_t hi = __shfl_down_sync(0xffffffffu, u[i], M + 1);
            const uint32_t lo = M == 0 ? u[i] : __shfl_up_sync(0xffffffffu, u[i], M == 0 ? 1 : M);
            dF[5 + i] = dF[4 + i] + hi - lo;
            dH[5 + i] = dH[4 + i] + (uint32_t)((int32_t)(hi - lo + 0x8000u) >> 16);
        }
#pragma unroll
        for (int i = 0; i < 4; i++) {  // column 4 - i -> 3 - i: column 8(l - M - 1) + 7 - i enters, column 8(l + M) + 7 - i leaves
            const uint32_t hi = M == 0 ? u[7 - i] : __shfl_down_sync(0xffffffffu, u[7 - i], M == 0 ? 1 : M);
            const uint32_t lo = __shfl_up_sync(0xffffffffu, u[7 - i], M + 1);
            dF[3 - i] = dF[4 - i] - hi + lo;
            dH[3 - i] = dH[4 - i] - (uint32_t)((int32_t)(hi - lo + 0x8000u) >> 16);
        }
        // every word of u carries the bias 0x80008000 (0x8000 on the odd field): 2K of them per window
        constexpr uint32_t BF = (uint32_t)(2 * K) * 0x80008000u, BH = (uint32_t)(2 * K) * 0x8000u;
#pragma unroll
        for (int j = 0; j < 8; j++) { F[j] += dF[j] - BF; Hh[j] += dH[j] - BH; }
    };
    // output row `it`: shift / cap / validity of the lane's 8 words, staged for the transposed store
    auto emit = [&](const int it) {
        const int srow = s_limy[it] - q.dmin - d;
        uint32_t w[8];
        if (__all_sync(0xffffffffu, min(thrmin, srow) >= 1)) {  // every cell of the warp's 256 x 2 cells is valid (the image interior)
#pragma unroll
            for (int j = 0; j < 8; j++) {
                const uint32_t chi = Hh[j], clo = F[j] - (chi << 16);
                const uint32_t c0 = min(clo >> q.shift, (uint32_t)q.cap), c1 = min(chi >> q.shift, (uint32_t)q.cap);
                w[j] = c1 * 65536u + c0;
            }
        } else {
#pragma unroll
            for (int j = 0; j < 8; j++) {
                const uint32_t chi = Hh[j], clo = F[j] - (chi << 16);
                uint32_t c0 = min(clo >> q.shift, (uint32_t)q.cap), c1 = min(chi >> q.shift, (uint32_t)q.cap);
                const int m = min(thr[j], srow);
                c0 = m >= 0 ? c0 : (uint32_t)q.cap;
                c1 = m >= 1 ? c1 : (uint32_t)q.cap;
                w[j] = c1 * 65536u + c0;
            }
        }
        // split barrier as in k_box_planar: announce this row, store the previous one
        if (it > 0) store_row(it - 1);
        // a lane's 32 bytes go out as two 16-byte stores; lanes 4..7 of every eight store their upper half first, so that the eight lanes
        // of a quarter-warp always hit eight different 16-byte bank groups (in lane order both halves would be 2-way conflicts)
        uint32_t* so = &s_out[it & 1][warp][lane * 8];
        const bool swz = (lane & 4) != 0;
        *reinterpret_cast<uint4*>(so + (swz ? 4 : 0)) = swz ? make_uint4(w[4], w[5], w[6], w[7]) : make_uint4(w[0], w[1], w[2], w[3]);
        *reinterpret_cast<uint4*>(so + (swz ? 0 : 4)) = swz ? make_uint4(w[0], w[1], w[2], w[3]) : make_uint4(w[4], w[5], w[6], w[7]);
        __syncwarp();
        if (lane == 0) asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar0 + 8 * (it & 1)) : "memory");
    };

    // ---- warm-up: updates 0 .. 2K-2 (rows entering, nothing leaving, no output), packed sums of `chunk` rows per horizontal pass ----
    {
        uint32_t acc[8];
#pragma unroll
        for (int j = 0; j < 8; j++) acc[j] = 0x80008000u;
        int cnt = 0;
        U32x8 a = ldg_stream_u256(pe, pol);
        for (int n = 0; n < 2 * K - 1; n++) {
            U32x8 b = a;
            if (n + 1 < 2 * K - 1) { pe += q.row_words; b = ldg_stream_u256(pe, pol); }
#pragma unroll
            for (int j = 0; j < 8; j++) acc[j] += a.v[j];
            if (++cnt == q.chunk || n + 1 == 2 * K - 1) {
                hpass(acc);
#pragma unroll
                for (int j = 0; j < 8; j++) acc[j] = 0x80008000u;
                cnt = 0;
            }
            a = b;
        }
    }
    // ---- steady state: update n = 2K-1+it adds physical row y0 + n, removes physical row y0 + n - 2K (zeros for it == 0), emits row it ----
    {
        const int R = y1 - y0;
        auto fetch = [&](const int it, U32x8& e, U32x8& l) {
            if (it < R) {
                pe += q.row_words;
                e = ldg_stream_u256(pe, pol);
                if (it > 0) l = ldg_stream_u256(pe - back, pol);
            }
        };
        auto row = [&](const int it, const U32x8& e, const U32x8& l) {
            uint32_t u[8];
#pragma unroll
            for (int j = 0; j < 8; j++) u[j] = e.v[j] - l.v[j] + 0x80008000u;
            hpass(u);
            emit(it);
        };
        // software pipeline: the loads of row it + PF are issued before row it is worked on; PF + 1 register buffers rotate by unrolling
        U32x8 be[PF + 1], bl[PF + 1];
#pragma unroll
        for (int i = 0; i <= PF; i++)
#pragma unroll
            for (int j = 0; j < 8; j++) { be[i].v[j] = 0; bl[i].v[j] = 0; }
#pragma unroll
        for (int i = 0; i < PF; i++) fetch(i, be[i], bl[i]);
        for (int it = 0; it < R; it += PF + 1) {
#pragma unroll
            for (int i = 0; i <= PF; i++) {
                if (it + i < R) {
                    fetch(it + i + PF, be[(i + PF) % (PF + 1)], bl[(i + PF) % (PF + 1)]);
                    row(it + i, be[i], bl[i]);
                }
            }
        }
        store_row(R - 1);  // the last row's deferred store
    }
    (void)N;
}

int sva_ap_prepare(sva_ctx* ctx);
int sva_ap_unpack(sva_ctx* ctx);

static int sva_launch_box_planar(sva_ctx* ctx) {
    const sva_params& p = ctx->prm;
    const int W = p.width, H = p.height, D = p.num_disp, k = p.win_half;
    BoxPParams q{};
    q.AP = ctx->AP.as<uint32_t>(); q.C = ctx->C.as<uint16_t>();
    q.W = W; q.H = H; q.D = D; q.k = k; q.kk = ctx->ap.padl; q.dmin = p.min_disp; q.shift = p.cost_shift; q.cap = p.cost_cap;
    for (int i = 0; i < p.n_pairs; i++) {
        int gx = p.pair_gx[i], gy = p.pair_gy[i];
        if (gx > 0) q.gxp = gx > q.gxp ? gx : q.gxp;
        if (gx < 0) q.gxn = -gx > q.gxn ? -gx : q.gxn;
        if (gy > 0) q.gyp = gy > q.gyp ? gy : q.gyp;
        if (gy < 0) q.gyn = -gy > q.gyn ? -gy : q.gyn;
    }
    q.txo = ctx->ap.txo; q.wp = ctx->ap.wp; q.row_words = (long long)ctx->ap.row_words;
    const int strips = ctx->ap.strips, dgroups = div_up(D, 16);
    // the register form of the horizontal sums needs win_half % 8 == 4 (k_box_planar_shfl); everything else takes the prefix table
    const bool shfl = ctx->tune_box_shfl && k % 8 == 4;
    auto shfl_kernel = [&](int occ) -> void (*)(BoxPParams) {
        switch (k) {
            case 4: return occ == 3 ? k_box_planar_shfl<4, 1, 3> : k_box_planar_shfl<4, 1, 2>;
            case 12: return occ == 3 ? k_box_planar_shfl<12, 1, 3> : k_box_planar_shfl<12, 1, 2>;
            case 20: return occ == 3 ? k_box_planar_shfl<20, 1, 3> : k_box_planar_shfl<20, 1, 2>;
            case 28: return occ == 3 ? k_box_planar_shfl<28, 1, 3> : k_box_planar_shfl<28, 1, 2>;
            case 36: return occ == 3 ? k_box_planar_shfl<36, 1, 3> : k_box_planar_shfl<36, 1, 2>;
            case 44: return occ == 3 ? k_box_planar_shfl<44, 1, 3> : k_box_planar_shfl<44, 1, 2>;
            default: return occ == 3 ? k_box_planar_shfl<52, 1, 3> : k_box_planar_shfl<52, 1, 2>;
        }
    };
    if (shfl) q.chunk = std::max(1, 32767 / (255 * p.n_pairs));
    q.ry0 = 0; q.ry1 = H;
    if (ctx->win_rows > 0) { q.ry0 = ctx->win_y0; q.ry1 = ctx->win_y0 + ctx->win_rows; }
    const int Hw = q.ry1 - q.ry0;
    // Row bands and CTAs per SM.  Every band re-reads 2k-1 warm-up rows (in the register form a third of an output row's DRAM traffic each,
    // and one horizontal pass per chunk), and the grid should fill whole waves of the resident CTAs.  The register form exists for 2 CTAs
    // per SM (up to 128 registers) and for 3 (80 registers, no spills): per row a CTA costs about the same either way and the SM's
    // throughput is shared, so the estimate is waves x CTAs per SM x rows marched per CTA — 3 per SM wins where 2 per SM would leave a
    // wave partly empty (c2, c4: 0.335 -> 0.309 ms, 0.617 -> 0.571 ms), 2 per SM where the bands are long anyway (c1, c3).
    void (*kern)(BoxPParams) = k_box_planar;
    const char* label = shfl ? "k_box_planar_shfl" : "k_box_planar";
    int bands = 1;
    double best = 1e30;
    const int per_band = strips * dgroups;
    for (int occ = 2; occ <= (shfl ? 3 : 2); occ++) {
        if (shfl && ctx->tune_box_occ && occ != ctx->tune_box_occ) continue;
        void (*cand)(BoxPParams) = shfl ? shfl_kernel(occ) : k_box_planar;
        int per_sm = occ;
        SVA_CUDA_OK(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, cand, 256, 0));
        if (per_sm < 1) per_sm = 1;
        const int slots = per_sm * ctx->sm_count;
        const double warm = shfl ? (2 * k - 1) / 3.0 + div_up(2 * k - 1, q.chunk) : (double)(2 * k - 1);
        for (int b = 1; b <= Hw && b <= 4096; b++) {
            const int rows = div_up(Hw, b);
            if (rows > BXP_MAX_BAND) continue;
            if (b > 1 && rows < k) break;
            const int nb = div_up(Hw, rows);
            const double cost = (double)div_up(nb * per_band, slots) * per_sm * (rows + warm + 8);
            if (cost < best) { best = cost; bands = nb; q.band_rows = rows; kern = cand; }
        }
    }
    if (ctx->tune_box_bands > 0) {
        const int rows = std::min(BXP_MAX_BAND, std::max(1, div_up(Hw, ctx->tune_box_bands)));
        q.band_rows = rows; bands = div_up(Hw, rows);
    }
    LaunchScope ls(ctx, label);
    kern<<<dim3(strips, dgroups, bands), 256, 0, ctx->stream>>>(q);
    SVA_CUDA_OK(ctx, cudaGetLastError());
    return SVA_OK;
}

int sva_run_box(sva_ctx* ctx, bool raw) {
    const sva_params& p = ctx->prm;
    size_t cells = (size_t)p.width * p.height * p.num_disp;
    if (raw) {  // RAW_U32 recomputation (download / test path): un-planarise A, then the general kernel
        SVA_TRY(ctx->reserve(ctx->Craw, cells * sizeof(uint32_t)));
        SVA_TRY(sva_ap_unpack(ctx));
        return sva_launch_box(ctx, ctx->A.as<uint16_t>(), ctx->Craw.p, p.width, p.height, p.num_disp, p.win_half, &p, true, true);
    }
    SVA_TRY(ctx->reserve(ctx->C, cells * sizeof(uint16_t)));
    SVA_TRY(sva_launch_box_planar(ctx));
    ctx->have_cost = true;
    return SVA_OK;
}
