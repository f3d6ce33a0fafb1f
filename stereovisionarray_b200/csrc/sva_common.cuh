// sva_common.cuh — context, error handling and small device helpers shared by the sm_100a kernels.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <set>
#include <string>
#include <vector>

#include "../../include/sva_c_api.h"

#define SVA_CUDA_OK(ctx, expr)                                                                         \
    do {                                                                                               \
        cudaError_t e__ = (expr);                                                                      \
        if (e__ != cudaSuccess) return (ctx)->fail(SVA_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(e__)); \
    } while (0)

#define SVA_TRY(expr)            \
    do {                         \
        int rc__ = (expr);       \
        if (rc__ != SVA_OK) return rc__; \
    } while (0)

// One growable device buffer.
struct DevBuf {
    void* p = nullptr;
    size_t bytes = 0;
    void* base = nullptr;  // start of the allocation when it carries guard bands (sva_debug_set_guard), else null
    template <typename T> T* as() const { return (T*)p; }
};

// Per-pair "line image": the other view re-laid out so that walking the disparity walks +g bytes along a row (k_ad.cu).
struct PairGeom {
    int32_t alpha, beta, base;  // byte offset of ref pixel (x,y) at delta=0:  base + x*alpha + y*beta
    int32_t g;                  // bytes per unit disparity (gcd(|gx|,|gy|))
    int32_t rows, pitch;        // line-image size
    int32_t a, b, u, v, cmin, tmin, pad;
    size_t offset;              // byte offset of this pair's line image inside ctx->lines
};

// Planar layout of the AD volume ("AP"): u16x2 words [Hp][D/2][Wp] — one plane per disparity PAIR and row, x fastest, with
// zero borders of padt rows above / below and padl columns left (k_ad.cu writes the interior, k_box.cu streams it).
struct ApGeom {
    int wp = 0, hp = 0, padl = 0, padt = 0;  // physical width / height in words / rows, left / top zero border
    int txo = 0, strips = 0;                 // k_box_planar: output columns per 256-column strip, strips per row
    size_t row_words = 0, words = 0;         // (D/2) * wp, hp * row_words
};

// Zero-bordered, 16-byte-pitched device copies of the views for the image-space AD kernel (k_ad2.cu).
struct Ad2Geom {
    int padx = 0, pady = 0, pp = 0, rows = 0;  // other views: left / top border, pitch, padded height
    int rp = 0, ref_rows = 0;                  // reference view: pitch, padded height
    size_t img_bytes = 0;                      // bytes per padded other view
};

// The per-frame input / output buffers of a context.  The streaming entry points (sva_stream_*) keep two such sets and swap them
// every frame, so frame t+1 uploads while frame t computes and frame t-1 downloads; the volumes (AP, C, S) are shared because the
// compute stages of consecutive frames run back to back on one stream.
struct IoSet {
    DevBuf pad_ref, pad_imgs, ref_img, other_imgs, lines, mask, disp, subpix;
    uint64_t ad2_zero_key = 0;
};

struct KernelTime {
    const char* name;
    cudaEvent_t beg, end;
};

struct sva_ctx {
    int device = 0;
    int sm_count = 148;
    cudaStream_t own_stream = nullptr;
    cudaStream_t stream = nullptr;
    cudaStream_t aux_stream = nullptr;  // second stream: the S memset of the next SGM runs next to K1a / K1b (sva_api.cu)
    cudaEvent_t ev_fork = nullptr, ev_zero = nullptr;
    bool s_prezeroed = false;  // S is being zeroed on aux_stream for the SGM of this whole-frame run (ev_zero marks the end)
    int tune_prezero = 1;      // SVA_PREZERO: overlap the S memset with K1a / K1b
    // ---- streaming pipeline (sva_stream_*) ----
    cudaStream_t h2d_stream = nullptr, d2h_stream = nullptr;
    cudaStream_t ad_stream = nullptr;   // K1a of frame t + 1 next to the SGM of frame t (sva_stream_submit)
    cudaEvent_t ev_ad = nullptr, ev_box = nullptr;
    bool ev_box_valid = false, in_stream_submit = false;
    int tune_stream_ad_ahead = 1;       // SVA_STREAM_AD_AHEAD
    cudaEvent_t ev_h2d[2] = {nullptr, nullptr}, ev_compute[2] = {nullptr, nullptr}, ev_done[2] = {nullptr, nullptr}, ev_mark = nullptr;
    IoSet alt;                 // the set not in use by the frame being submitted
    int64_t stream_ticket = 0; // next ticket
    std::string err;
    uint64_t launches = 0;

    // ---- resident frame state (volume mode) ----
    bool have_frame = false, have_ad = false, have_cost = false, have_sgm = false, have_disp = false;
    sva_params prm{};
    sva_params up_prm{};        // parameters of the last upload: what the view staging was laid out for
    bool ad_params_ok = false;  // prm still matches that staging (sva_frame_set_params may break it; SVA_STAGE_AD then refuses)
    int ad_y0 = 0, ad_y1 = 0, cost_y0 = 0, cost_y1 = 0;  // image rows of A / C that hold the current frame (row-block runs fill only part)
    int pair_begin = 0, pair_end = 0;
    bool has_mask = false;
    bool debug_store_full_s = false;
    int tune_sgm_split = 1;       // SVA_SGM_SPLIT: 8 paths as three launches (down-sweeping, up-sweeping, horizontal; default) or, 0, as one
    int tune_sgm_hstore = 2;      // SVA_SGM_HSTORE: 1 = the first horizontal direction initialises S with plain stores (no memset) and the second accumulates;
                                  // 2 (default) = and the second runs on the second stream next to the first row-sweeping group where the launches are not
                                  // paced; 3 = always next to it; 0 = S zeroed by a memset next to K1, both horizontal directions in one launch
    int tune_sgm_pace = -1;       // SVA_SGM_PACE: keep all CTAs of a row-sweeping launch within pace_window rounds (of 9 rows) of each other.
                                  // -1 = automatic: on when one image row of C + S (W*D*4 bytes) is 768 KB or more.  The three directions of such a
                                  // launch share C and S lines in L2 only while their rows stay within the L2-resident window; unpaced drift is harmless
                                  // at c1 (0.66 MB per row: 0.277 ms unpaced, 0.283 paced) and costly at c4 (1.47 MB per row: 1.355 -> 0.925 ms paced).
    int tune_sgm_pace_window = 2; // SVA_SGM_PACE_WINDOW: rounds of 9 rows
    int tune_sgm_bulk = 0;        // SVA_SGM_BULK: 1 = C streams in by the TMA engine's bulk copies + mbarriers, 2 = and S is accumulated by bulk reduces;
                                  // 0 (default, fastest measured) = per-lane cp.async / RED
    int tune_sgm_diag_split = 1;  // SVA_SGM_DIAG_SPLIT: diagonal lines run the march that is split at the wrap events (no per-step wrap logic)
    int tune_ad_gather = 0;       // SVA_AD_GATHER=1: force the line-image gather AD kernel (k_ad.cu) even where the image-space kernel applies
    int tune_ad_set = 1;          // SVA_AD_SET: use the AD kernel compiled for the frame's pair set where one exists (0 = always the generic kernel)
    int tune_ad_th = 0;           // SVA_AD_TH: rows per tile of the image-space AD kernel (0 = chosen per launch, k_ad2.cu)
    int tune_box_l2 = 0;          // SVA_BOX_L2: K1b's entering rows stay in L2 (evict_last) for their second read as leaving rows (evict_first, like the C stores)
    int tune_box_occ = 0;         // SVA_BOX_OCC: CTAs per SM K1b is compiled for (2: up to 128 registers, 3: 80; 0 = chosen per launch)
    int tune_box_bands = 0;       // SVA_BOX_BANDS: row bands of K1b (0 = chosen per launch)
    int tune_box_shfl = 1;        // SVA_BOX_SHFL: K1b's horizontal window sums by warp shuffles where win_half % 8 == 4 (0 = the shared-memory prefix table)
    int tune_wta_seg = -1;        // SVA_WTA_SEG: K3 as a register march over row segments of this many pixels (-1 = chosen per frame: 96 or 160;
                                  // 0 = the shared-memory tile kernel)
    uint32_t sgm_dir_mask_override = 0;  // tests: run exactly these directions as accumulate passes (no final pass)
    PairGeom geom[SVA_MAX_PAIRS];
    DevBuf ref_img, other_imgs, lines, mask, A, AP, C, Craw, S, disp, subpix, other_d, scratch, scratch2, pace_buf;
    DevBuf pad_imgs, pad_ref, comm_scratch, census, tex_img, sgm_state;
    unsigned long long tex = 0;  // cudaTextureObject_t over tex_img (K0's source view, k_misc.cu)
    uint64_t tex_key = 0;
    // ---- multi-GPU (sva_dist.cu) ----
    void* comm = nullptr;        // ncclComm_t (sva_comm_init)
    int comm_rank = 0, comm_world = 1;
    void* rows_link = nullptr;   // RowsLink: peer-mapped state buffers and flags of the row-block pipeline (sva_rows_open)
    Ad2Geom ad2;
    uint64_t ad2_zero_key = 0;
    bool use_ad2 = false;      // this frame's AD volume comes from k_ad_tile (all pair offsets within +-2) instead of the line-image gather
    ApGeom ap;
    uint64_t ap_zero_key = 0;  // geometry + buffer the zero borders of AP were last established for
    DevBuf staging_host;  // pinned host staging for image uploads / result downloads
    int win_y0 = 0, win_rows = 0;  // row-block pipeline: K1a / K1b compute only what image rows [win_y0, win_y0 + win_rows) need (0 rows = whole frame)
    bool guard = false;   // debug: new device allocations get canary bands on both sides and a poisoned interior (sva_debug_set_guard)
    void device_bufs(std::vector<DevBuf*>& out);
    void release(DevBuf& b);

    // ---- per-kernel timing of the last run ----
    bool timing = false;
    std::vector<KernelTime> ktimes;
    std::vector<cudaEvent_t> event_pool;
    size_t events_used = 0;

    std::set<std::string> names;  // timing labels built at run time (node-based: the c_str() pointers stay valid)
    const char* intern(const std::string& s) { return names.insert(s).first->c_str(); }
    int fail(int code, const std::string& msg) {
        err = msg;
        return code;
    }
    int reserve(DevBuf& b, size_t bytes);
    int reserve_pinned(DevBuf& b, size_t bytes);
    void time_begin(const char* name);
    void time_end();
};

// RAII-ish helper: records an event pair around a kernel when ctx->timing is on, and counts the launch.
struct LaunchScope {
    sva_ctx* c;
    LaunchScope(sva_ctx* ctx, const char* name) : c(ctx) {
        c->launches++;
        if (c->timing) c->time_begin(name);
    }
    ~LaunchScope() {
        if (c->timing) c->time_end();
    }
};

static inline int div_up(int a, int b) { return (a + b - 1) / b; }

// an environment switch's value as a whole number in [lo, hi]; false for text, overflow or a value outside (sva_ctx.cu)
bool sva_parse_env_int(const char* s, long long lo, long long hi, long long* out);

#ifdef __CUDACC__
// streaming (read-once) global loads: bypass L1 allocation
__device__ __forceinline__ uint32_t ldg_stream_u32(const void* p) {
    uint32_t v;
    asm volatile("ld.global.nc.L1::no_allocate.u32 %0, [%1];" : "=r"(v) : "l"(p));
    return v;
}
__device__ __forceinline__ uint2 ldg_stream_u64(const void* p) {
    uint2 v;
    asm volatile("ld.global.nc.L1::no_allocate.v2.u32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "l"(p));
    return v;
}
__device__ __forceinline__ uint4 ldg_stream_u128(const void* p) {
    uint4 v;
    asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p));
    return v;
}
// 32 bytes per lane in ONE instruction (LDG.E.256, sm_100): a warp-load covers 1 KB of whole sectors.  `policy` is an L2 eviction
// policy word from l2_policy_* below.  The address must be 32-byte aligned.
struct U32x8 { uint32_t v[8]; };
__device__ __forceinline__ U32x8 ldg_stream_u256(const void* p, const unsigned long long policy) {
    U32x8 r;
    asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.v8.u32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8], %9;"
                 : "=r"(r.v[0]), "=r"(r.v[1]), "=r"(r.v[2]), "=r"(r.v[3]), "=r"(r.v[4]), "=r"(r.v[5]), "=r"(r.v[6]), "=r"(r.v[7])
                 : "l"(p), "l"(policy));
    return r;
}
__device__ __forceinline__ unsigned long long l2_policy_evict_last() {
    unsigned long long pol;
    asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(pol));
    return pol;
}
__device__ __forceinline__ unsigned long long l2_policy_evict_first() {
    unsigned long long pol;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
    return pol;
}
__device__ __forceinline__ unsigned long long l2_policy_evict_normal() {
    unsigned long long pol;
    asm volatile("createpolicy.fractional.L2::evict_normal.b64 %0, 1.0;" : "=l"(pol));
    return pol;
}
__device__ __forceinline__ void stg_u128_hint(void* p, const uint4& v, const unsigned long long policy) {
    asm volatile("st.global.L2::cache_hint.v4.u32 [%0], {%1, %2, %3, %4}, %5;" ::"l"(p), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w), "l"(policy) : "memory");
}
#endif
