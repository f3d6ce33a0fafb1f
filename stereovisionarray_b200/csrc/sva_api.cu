// sva_api.cu — extern "C" entry points of the volume-mode pipeline (staged / device-resident and host-buffer forms).
#include <algorithm>
#include <cstring>

#include <nvtx3/nvToolsExt.h>  // header-only: ranges are no-ops unless a profiler injects itself

#include "sva_common.cuh"

// one NVTX range per pipeline stage (SURVEY §5): nsys / ncu --nvtx group the kernels by the stage that launched them
struct NvtxRange {
    explicit NvtxRange(const char* name) { nvtxRangePushA(name); }
    ~NvtxRange() { nvtxRangePop(); }
};

int sva_build_line_images(sva_ctx* ctx);
int sva_run_ad(sva_ctx* ctx);
int sva_run_ad_census(sva_ctx* ctx);
int sva_run_box(sva_ctx* ctx, bool raw);
int sva_run_sgm(sva_ctx* ctx);
int sva_sgm_regs_per_lane(int D);
int sva_ap_prepare(sva_ctx* ctx);
bool sva_ad2_usable(const sva_params& p);
int sva_ad2_prepare(sva_ctx* ctx);
uint8_t* sva_ad2_view_origin(sva_ctx* ctx, int k);
int sva_run_ad2(sva_ctx* ctx);
int sva_run_sgm_dirs(sva_ctx* ctx, const uint16_t* Cext, int c_ds, uint32_t dir_mask, int rows_alloc);
int sva_run_wta_rows(sva_ctx* ctx, const uint16_t* vol, int y0, int rows);
int sva_run_sgm_rows(sva_ctx* ctx, int group, int y0, int rows, const uint16_t* state_in, uint16_t* state_out);
int sva_ap_unpack(sva_ctx* ctx);
int sva_stream_enqueue(sva_ctx* c, const sva_params* p, const sva_image_u8* ref, const sva_image_u8* others, const sva_image_u8* mask,
                       cudaMemcpyKind view_kind, uint16_t* out_disp, float* out_subpix, int64_t* out_ticket);

// (also used by sva_depth_groups, sva_groups.cu: every group's derived parameters are checked before anything is enqueued)
int check_params(sva_ctx* c, const sva_params* p) {
    if (!p) return c->fail(SVA_ERR_BAD_ARG, "null params");
    if (p->width < 8 || p->height < 8) return c->fail(SVA_ERR_BAD_ARG, "image smaller than 8x8");
    if (p->num_disp < 8 || p->num_disp > 256 || p->num_disp % 8) return c->fail(SVA_ERR_BAD_ARG, "num_disp must be a multiple of 8 in 8..256");
    if (p->min_disp < 0 || p->min_disp > 4096) return c->fail(SVA_ERR_BAD_ARG, "min_disp must be in 0..4096");
    if (p->win_half < 1 || p->win_half > 56) return c->fail(SVA_ERR_BAD_ARG, "win_half must be in 1..56");
    if (p->n_pairs < 1 || p->n_pairs > SVA_MAX_PAIRS) return c->fail(SVA_ERR_BAD_ARG, "n_pairs must be in 1..32");
    if (p->cost_cap < 1 || p->cost_cap > SVA_COST_CAP_MAX || p->cost_shift < 0 || p->cost_shift > 31) return c->fail(SVA_ERR_BAD_ARG, "bad cost_cap / cost_shift");
    if (p->p1 < 0 || p->p2 < p->p1 || p->p2 > 4095) return c->fail(SVA_ERR_BAD_ARG, "need 0 <= p1 <= p2 <= 4095");
    if (p->n_paths != 0 && p->n_paths != 4 && p->n_paths != 8) return c->fail(SVA_ERR_BAD_ARG, "n_paths must be 0, 4 or 8");
    if (p->lr_gx < -1 || p->lr_gx > 1) return c->fail(SVA_ERR_BAD_ARG, "lr_gx must be -1, 0 or +1");
    if (sva_sgm_regs_per_lane(p->num_disp) == 0) return c->fail(SVA_ERR_BAD_ARG, "unsupported num_disp");
    if (p->reserved[0] != SVA_COST_SAD && p->reserved[0] != SVA_COST_CENSUS) return c->fail(SVA_ERR_BAD_ARG, "unknown cost mode (reserved[0])");
    for (int i = 1; i < 8; i++) if (p->reserved[i] != 0) return c->fail(SVA_ERR_BAD_ARG, "reserved parameter fields must be zero");
    // exact u32 box sums: 4k^2 * 255 * n_pairs must fit (census cells are smaller still)
    if (4.0 * p->win_half * p->win_half * 255.0 * p->n_pairs > 4.0e9) return c->fail(SVA_ERR_BAD_ARG, "window sum overflows u32");
    // the marches index the volumes with 32-bit element cursors
    if ((double)p->width * p->height * p->num_disp >= 4294967296.0) return c->fail(SVA_ERR_BAD_ARG, "frame too large: width * height * num_disp must be below 2^32");
    return SVA_OK;
}

static int check_image(sva_ctx* c, const sva_image_u8* im, int W, int H, const char* what) {
    if (!im || !im->data) return c->fail(SVA_ERR_BAD_ARG, std::string("null image: ") + what);
    if (im->cols != W || im->rows != H || im->step < (size_t)W) return c->fail(SVA_ERR_BAD_ARG, std::string("image size / step mismatch: ") + what);
    return SVA_OK;
}

// rows [b0, b1) join the interval [a0, a1) a volume already holds of this frame when they touch it, and replace it otherwise
static void merge_rows(int& a0, int& a1, int b0, int b1) {
    if (a1 <= a0 || b0 > a1 || b1 < a0) { a0 = b0; a1 = b1; return; }
    a0 = std::min(a0, b0); a1 = std::max(a1, b1);
}

// (also used by sva_rows_stream_submit, sva_dist.cu: a frame is refused before anything of it is enqueued)
int check_frame_args(sva_ctx* c, const sva_params* p, const sva_image_u8* ref, const sva_image_u8* others, const sva_image_u8* mask) {
    SVA_TRY(check_params(c, p));
    const int W = p->width, H = p->height;
    SVA_TRY(check_image(c, ref, W, H, "ref"));
    if (!others) return c->fail(SVA_ERR_BAD_ARG, "null others");
    for (int i = 0; i < p->n_pairs; i++) SVA_TRY(check_image(c, &others[i], W, H, "other view"));
    if (mask) SVA_TRY(check_image(c, mask, W, H, "mask"));
    return SVA_OK;
}

// The copy part of an upload: the views into the staging of the kernels that will read them, from host memory (view_kind =
// cudaMemcpyHostToDevice) or from device memory (cudaMemcpyDeviceToDevice: an array frame's camera stack, sva_depth_groups); the mask is
// always a host buffer.  In census mode with ctx->sig_stack set, K1a reads the stack's signatures and no view is staged.
static int stage_frame(sva_ctx* c, const sva_params* p, const sva_image_u8* ref, const sva_image_u8* others, const sva_image_u8* mask, cudaMemcpyKind view_kind) {
    NvtxRange range("sva:upload");
    SVA_CUDA_OK(c, cudaSetDevice(c->device));
    SVA_TRY(check_frame_args(c, p, ref, others, mask));
    const int W = p->width, H = p->height;
    c->prm = *p;
    c->up_prm = *p;  // the view staging (zero borders, phi column offsets, line images) is laid out for THIS disparity reach and these pairs
    c->ad_params_ok = true;
    c->win_y0 = 0; c->win_rows = 0;
    c->pair_begin = 0; c->pair_end = p->n_pairs;
    c->have_frame = c->have_ad = c->have_cost = c->have_sgm = c->have_disp = false;
    c->s_prezeroed = false;
    c->ad_y0 = c->ad_y1 = c->cost_y0 = c->cost_y1 = 0;
    const size_t img = (size_t)W * H;
    const bool census = p->reserved[0] == SVA_COST_CENSUS;
    c->use_ad2 = sva_ad2_usable(*p) && !c->tune_ad_gather && !census;
    if (c->use_ad2) {
        // image-space AD kernel: the views go straight into zero-bordered, 16-byte-pitched device copies
        SVA_TRY(sva_ad2_prepare(c));
        SVA_CUDA_OK(c, cudaMemcpy2DAsync(c->pad_ref.p, c->ad2.rp, ref->data, ref->step, W, H, view_kind, c->stream));
        for (int i = 0; i < p->n_pairs; i++)
            SVA_CUDA_OK(c, cudaMemcpy2DAsync(sva_ad2_view_origin(c, i), c->ad2.pp, others[i].data, others[i].step, W, H, view_kind, c->stream));
    } else if (!(census && c->sig_stack)) {
        SVA_TRY(c->reserve(c->ref_img, img));
        SVA_TRY(c->reserve(c->other_imgs, img * p->n_pairs));
        SVA_CUDA_OK(c, cudaMemcpy2DAsync(c->ref_img.p, W, ref->data, ref->step, W, H, view_kind, c->stream));
        for (int i = 0; i < p->n_pairs; i++)
            SVA_CUDA_OK(c, cudaMemcpy2DAsync(c->other_imgs.as<uint8_t>() + img * i, W, others[i].data, others[i].step, W, H, view_kind, c->stream));
    }
    c->has_mask = mask != nullptr;
    if (mask) {
        SVA_TRY(c->reserve(c->mask, img));
        SVA_CUDA_OK(c, cudaMemcpy2DAsync(c->mask.p, W, mask->data, mask->step, W, H, cudaMemcpyHostToDevice, c->stream));
    }
    if (!c->use_ad2 && !census) SVA_TRY(sva_build_line_images(c));
    c->have_frame = true;
    return SVA_OK;
}

extern "C" {

int sva_frame_upload(sva_ctx* c, const sva_params* p, const sva_image_u8* ref, const sva_image_u8* others, const sva_image_u8* mask) {
    if (!c) return SVA_ERR_BAD_ARG;
    return stage_frame(c, p, ref, others, mask, cudaMemcpyHostToDevice);
}

int sva_frame_set_pair_range(sva_ctx* c, int32_t b, int32_t e) {
    if (!c || !c->have_frame) return c ? c->fail(SVA_ERR_STATE, "no frame uploaded") : SVA_ERR_BAD_ARG;
    if (b < 0 || e > c->prm.n_pairs || b > e) return c->fail(SVA_ERR_BAD_ARG, "bad pair range");
    c->pair_begin = b; c->pair_end = e;
    return SVA_OK;
}

int sva_frame_set_debug(sva_ctx* c, int32_t store_full_s, uint32_t sgm_dir_mask) {
    if (!c) return SVA_ERR_BAD_ARG;
    c->debug_store_full_s = store_full_s != 0;
    c->sgm_dir_mask_override = sgm_dir_mask;
    return SVA_OK;
}

// Whole-frame runs zero the aggregation volume S on the second stream while K1a / K1b (bound by the integer pipe, not by HBM) run on
// the main one; sva_run_sgm joins the event instead of issuing its own memset.
static int prezero_s(sva_ctx* c) {
    const sva_params& p = c->prm;
    c->s_prezeroed = false;
    if (p.n_paths == 0 || c->sgm_dir_mask_override || !c->tune_prezero) return SVA_OK;
    if (p.n_paths == 8) return SVA_OK;  // S is written, not accumulated, by the first SGM launch
    const size_t bytes = (size_t)p.width * p.height * p.num_disp * sizeof(uint16_t);
    SVA_TRY(c->reserve(c->S, bytes + 64));
    if (!c->aux_stream) {
        SVA_CUDA_OK(c, cudaStreamCreateWithFlags(&c->aux_stream, cudaStreamNonBlocking));
        SVA_CUDA_OK(c, cudaEventCreateWithFlags(&c->ev_fork, cudaEventDisableTiming));
    }
    if (!c->ev_zero) SVA_CUDA_OK(c, cudaEventCreateWithFlags(&c->ev_zero, cudaEventDisableTiming));
    SVA_CUDA_OK(c, cudaEventRecord(c->ev_fork, c->stream));            // after the previous frame's last reader of S
    SVA_CUDA_OK(c, cudaStreamWaitEvent(c->aux_stream, c->ev_fork, 0));
    SVA_CUDA_OK(c, cudaMemsetAsync(c->S.p, 0, bytes, c->aux_stream));
    SVA_CUDA_OK(c, cudaEventRecord(c->ev_zero, c->aux_stream));
    c->s_prezeroed = true;
    return SVA_OK;
}

static int run_stage(sva_ctx* c, int stage) {
    if (!c->in_stream_submit) c->ev_box_valid = false;  // work outside the capture stream uses AP too: the next streamed K1a waits for all of it
    NvtxRange range(stage == SVA_STAGE_AD ? "sva:K1a_ad_volume" : stage == SVA_STAGE_BOX ? "sva:K1b_box_cost" : stage == SVA_STAGE_SGM ? "sva:K2_sgm+K3_wta" : "sva:frame");
    switch (stage) {
        case SVA_STAGE_AD: {
            if (!c->have_frame) return c->fail(SVA_ERR_STATE, "no frame uploaded");
            if (!c->ad_params_ok)
                return c->fail(SVA_ERR_STATE, "sva_frame_set_params changed the pairs / disparity reach the views were staged for at upload: upload the frame again before SVA_STAGE_AD");
            SVA_TRY(c->prm.reserved[0] == SVA_COST_CENSUS ? sva_run_ad_census(c) : c->use_ad2 ? sva_run_ad2(c) : sva_run_ad(c));
            // rows of A that now hold this frame: the block's rows +- win_half (clipped), or everything
            const int H = c->prm.height, k = c->prm.win_half;
            if (c->pair_begin != 0 || c->pair_end != c->prm.n_pairs) c->ad_y0 = c->ad_y1 = 0;  // a pair-range partial replaces what A held
            merge_rows(c->ad_y0, c->ad_y1, c->win_rows > 0 ? std::max(0, c->win_y0 - k) : 0, c->win_rows > 0 ? std::min(H, c->win_y0 + c->win_rows + k) : H);
            return SVA_OK;
        }
        case SVA_STAGE_BOX: {
            if (!c->have_ad) return c->fail(SVA_ERR_STATE, "AD volume not computed");
            const int H = c->prm.height, k = c->prm.win_half;
            const int y0 = c->win_rows > 0 ? c->win_y0 : 0, y1 = c->win_rows > 0 ? c->win_y0 + c->win_rows : H;
            if (c->ad_y1 > c->ad_y0 && (std::max(0, y0 - k) < c->ad_y0 || std::min(H, y1 + k) > c->ad_y1))  // (an externally reduced A has no interval: ad_y0 == ad_y1)
                return c->fail(SVA_ERR_STATE, "the AD volume does not cover the rows this box filter reads: run SVA_STAGE_AD for the current row block");
            SVA_TRY(sva_run_box(c, false));
            merge_rows(c->cost_y0, c->cost_y1, y0, y1);
            return SVA_OK;
        }
        case SVA_STAGE_SGM:
            if (!c->have_cost) return c->fail(SVA_ERR_STATE, "cost volume not computed");
            if (c->win_rows > 0)  // only the block's rows of the cost volume exist
                return c->fail(SVA_ERR_STATE, "a row block is active (sva_frame_rows_begin): use sva_frame_sgm_rows, or upload the frame again for a whole-frame run");
            if (c->cost_y0 > 0 || c->cost_y1 < c->prm.height)
                return c->fail(SVA_ERR_STATE, "the cost volume holds only a row block of this frame: run SVA_STAGE_AD / SVA_STAGE_BOX on the whole frame first");
            return sva_run_sgm(c);
        case SVA_STAGE_ALL: {
            SVA_TRY(prezero_s(c));
            int rc = run_stage(c, SVA_STAGE_AD);
            if (rc == SVA_OK) rc = run_stage(c, SVA_STAGE_BOX);
            if (rc == SVA_OK) rc = run_stage(c, SVA_STAGE_SGM);
            if (rc != SVA_OK) c->s_prezeroed = false;  // nobody will join ev_zero for this run
            return rc;
        }
        default: return c->fail(SVA_ERR_BAD_ARG, "unknown stage");
    }
}

int sva_frame_run(sva_ctx* c, int32_t stage) {
    if (!c) return SVA_ERR_BAD_ARG;
    SVA_CUDA_OK(c, cudaSetDevice(c->device));
    return run_stage(c, stage);
}

int sva_frame_time(sva_ctx* c, int32_t stage, int32_t iters, float* out_ms) {
    if (!c || !out_ms || iters < 1) return SVA_ERR_BAD_ARG;
    SVA_CUDA_OK(c, cudaSetDevice(c->device));
    cudaEvent_t e0, e1;
    SVA_CUDA_OK(c, cudaEventCreate(&e0));
    SVA_CUDA_OK(c, cudaEventCreate(&e1));
    SVA_CUDA_OK(c, cudaStreamSynchronize(c->stream));
    SVA_CUDA_OK(c, cudaEventRecord(e0, c->stream));
    int rc = SVA_OK;
    for (int i = 0; i < iters && rc == SVA_OK; i++) rc = run_stage(c, stage);
    SVA_CUDA_OK(c, cudaEventRecord(e1, c->stream));
    SVA_CUDA_OK(c, cudaEventSynchronize(e1));
    SVA_CUDA_OK(c, cudaEventElapsedTime(out_ms, e0, e1));
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    return rc;
}

/* like sva_frame_time, with a CUDA-event pair around every kernel: per distinct kernel name the summed time and launch count */
int sva_frame_time_detailed(sva_ctx* c, int32_t stage, int32_t iters, float* out_total_ms, const char** names, float* sum_ms, int32_t* counts, int32_t cap) {
    if (!c || !out_total_ms || iters < 1) return SVA_ERR_BAD_ARG;
    SVA_CUDA_OK(c, cudaSetDevice(c->device));
    c->ktimes.clear(); c->events_used = 0;
    cudaEvent_t e0, e1;
    SVA_CUDA_OK(c, cudaEventCreate(&e0));
    SVA_CUDA_OK(c, cudaEventCreate(&e1));
    SVA_CUDA_OK(c, cudaStreamSynchronize(c->stream));
    c->timing = true;
    SVA_CUDA_OK(c, cudaEventRecord(e0, c->stream));
    int rc = SVA_OK;
    for (int i = 0; i < iters && rc == SVA_OK; i++) rc = run_stage(c, stage);
    SVA_CUDA_OK(c, cudaEventRecord(e1, c->stream));
    c->timing = false;
    SVA_CUDA_OK(c, cudaEventSynchronize(e1));
    SVA_CUDA_OK(c, cudaEventElapsedTime(out_total_ms, e0, e1));
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    if (rc != SVA_OK) return rc;
    int n = 0;
    for (const KernelTime& kt : c->ktimes) {
        float ms = 0;
        SVA_CUDA_OK(c, cudaEventElapsedTime(&ms, kt.beg, kt.end));
        int j = 0;
        for (; j < n; j++) if (names[j] == kt.name) break;
        if (j == n) { if (n >= cap) continue; names[n] = kt.name; sum_ms[n] = 0; counts[n] = 0; n++; }
        sum_ms[j] += ms; counts[j]++;
    }
    return n;
}

/* CUDA-event stopwatch on the ctx stream, for timing a sequence of host-buffer calls (the e2e path) on the device clock */
int sva_timer_start(sva_ctx* c) {
    if (!c) return SVA_ERR_BAD_ARG;
    SVA_CUDA_OK(c, cudaSetDevice(c->device));
    while (c->event_pool.size() < 2) { cudaEvent_t e; SVA_CUDA_OK(c, cudaEventCreate(&e)); c->event_pool.push_back(e); }
    SVA_CUDA_OK(c, cudaStreamSynchronize(c->stream));
    SVA_CUDA_OK(c, cudaEventRecord(c->event_pool[0], c->stream));
    return SVA_OK;
}
int sva_timer_stop(sva_ctx* c, float* out_ms) {
    if (!c || !out_ms || c->event_pool.size() < 2) return SVA_ERR_BAD_ARG;
    SVA_CUDA_OK(c, cudaEventRecord(c->event_pool[1], c->stream));
    SVA_CUDA_OK(c, cudaEventSynchronize(c->event_pool[1]));
    SVA_CUDA_OK(c, cudaEventElapsedTime(out_ms, c->event_pool[0], c->event_pool[1]));
    return SVA_OK;
}

int sva_frame_kernel_times(sva_ctx* c, int32_t stage, const char** names, float* ms, int32_t cap) {
    if (!c) return SVA_ERR_BAD_ARG;
    SVA_CUDA_OK(c, cudaSetDevice(c->device));
    c->ktimes.clear(); c->events_used = 0;
    c->timing = true;
    int rc = run_stage(c, stage);
    c->timing = false;
    if (rc != SVA_OK) return rc;
    SVA_CUDA_OK(c, cudaStreamSynchronize(c->stream));
    int n = (int)c->ktimes.size();
    for (int i = 0; i < n && i < cap; i++) {
        if (names) names[i] = c->ktimes[i].name;
        if (ms) SVA_CUDA_OK(c, cudaEventElapsedTime(&ms[i], c->ktimes[i].beg, c->ktimes[i].end));
    }
    return n;
}

static int download(sva_ctx* c, bool have, const DevBuf& b, void* out, size_t bytes, const char* what) {
    if (!c || !out) return SVA_ERR_BAD_ARG;
    if (!have) return c->fail(SVA_ERR_STATE, std::string("not computed yet: ") + what);
    SVA_CUDA_OK(c, cudaSetDevice(c->device));
    SVA_CUDA_OK(c, cudaMemcpyAsync(out, b.p, bytes, cudaMemcpyDeviceToHost, c->stream));
    SVA_CUDA_OK(c, cudaStreamSynchronize(c->stream));
    return SVA_OK;
}

static size_t cells(const sva_ctx* c) { return (size_t)c->prm.width * c->prm.height * c->prm.num_disp; }

int sva_frame_download_ad(sva_ctx* c, uint16_t* out) {
    if (!c || !out) return SVA_ERR_BAD_ARG;
    if (!c->have_ad) return c->fail(SVA_ERR_STATE, "not computed yet: AD volume");
    SVA_CUDA_OK(c, cudaSetDevice(c->device));
    SVA_TRY(sva_ap_unpack(c));  // the device volume is planar (ApGeom); the C ABI hands out [H][W][D]
    return download(c, true, c->A, out, cells(c) * 2, "AD volume");
}
int sva_frame_download_cost(sva_ctx* c, uint16_t* out) { return download(c, c && c->have_cost, c->C, out, cells(c) * 2, "cost volume"); }
int sva_frame_download_sgm(sva_ctx* c, uint16_t* out) { return download(c, c && c->have_sgm, c->S, out, cells(c) * 2, "aggregated volume"); }
int sva_frame_download_raw_cost(sva_ctx* c, uint32_t* out) {
    if (!c || !out) return SVA_ERR_BAD_ARG;
    if (!c->have_ad) return c->fail(SVA_ERR_STATE, "AD volume not computed");
    SVA_CUDA_OK(c, cudaSetDevice(c->device));
    SVA_TRY(sva_run_box(c, true));
    return download(c, true, c->Craw, out, cells(c) * 4, "raw cost");
}
int sva_frame_download_disparity(sva_ctx* c, uint16_t* out_disp, float* out_sub) {
    if (!c || !out_disp) return SVA_ERR_BAD_ARG;
    if (!c->have_disp) return c->fail(SVA_ERR_STATE, "disparity not computed");
    SVA_CUDA_OK(c, cudaSetDevice(c->device));
    size_t px = (size_t)c->prm.width * c->prm.height;
    SVA_CUDA_OK(c, cudaMemcpyAsync(out_disp, c->disp.p, px * 2, cudaMemcpyDeviceToHost, c->stream));
    if (out_sub) SVA_CUDA_OK(c, cudaMemcpyAsync(out_sub, c->subpix.p, px * 4, cudaMemcpyDeviceToHost, c->stream));
    SVA_CUDA_OK(c, cudaStreamSynchronize(c->stream));
    return SVA_OK;
}

int sva_frame_ad_device_ptr(sva_ctx* c, void** out_ptr, size_t* out_bytes) {
    if (!c || !out_ptr || !out_bytes) return SVA_ERR_BAD_ARG;
    if (!c->have_frame) return c->fail(SVA_ERR_STATE, "no frame uploaded");
    SVA_CUDA_OK(c, cudaSetDevice(c->device));
    SVA_TRY(sva_ap_prepare(c));  // planar layout incl. its zero borders: a cross-GPU sum is element-wise, so the layout does not matter
    *out_ptr = c->AP.p; *out_bytes = c->ap.words * 4;
    return SVA_OK;
}
/* after an external (cross-GPU) reduction wrote the full A volume into the buffer above */
int sva_frame_mark_ad_ready(sva_ctx* c) {
    if (!c || !c->have_frame) return SVA_ERR_BAD_ARG;
    c->have_ad = true;
    c->ad_y0 = c->ad_y1 = 0;  // written by the caller: no interval to check
    return SVA_OK;
}

int sva_depth_from_array(sva_ctx* c, const sva_params* p, const sva_image_u8* ref, const sva_image_u8* others, const sva_image_u8* mask,
                         uint16_t* out_disp, float* out_subpix) {
    if (!c || !out_disp) return SVA_ERR_BAD_ARG;
    SVA_TRY(sva_frame_upload(c, p, ref, others, mask));
    SVA_TRY(run_stage(c, SVA_STAGE_ALL));
    return sva_frame_download_disparity(c, out_disp, out_subpix);
}

/* ---- multi-GPU building blocks: disparity-slice / direction / row sharding of ONE frame (DESIGN.md §7) ----------------------------
 * rank r uploads the frame with num_disp = D/G, min_disp = dmin + r*D/G and runs STAGE_AD + STAGE_BOX: its slice of the cost volume
 * (no cross-GPU reduction at all).  The slices are all-gathered into a slice-major volume [G][H][W][D/G]; every rank switches to the full
 * disparity range (sva_frame_set_params), aggregates ITS directions on the gathered volume (sva_frame_sgm_directions) and the partial
 * sums are reduce-scattered by row blocks; each rank then runs K3 on its rows (sva_frame_wta_rows). */
int sva_frame_cost_device_ptr(sva_ctx* c, void** out_ptr, size_t* out_bytes) {
    if (!c || !out_ptr || !out_bytes) return SVA_ERR_BAD_ARG;
    if (!c->have_cost) return c->fail(SVA_ERR_STATE, "cost volume not computed");
    *out_ptr = c->C.p; *out_bytes = cells(c) * 2;
    return SVA_OK;
}

int sva_frame_set_params(sva_ctx* c, const sva_params* p) {
    if (!c) return SVA_ERR_BAD_ARG;
    if (!c->have_frame) return c->fail(SVA_ERR_STATE, "no frame uploaded");
    SVA_TRY(check_params(c, p));
    if (p->width != c->prm.width || p->height != c->prm.height) return c->fail(SVA_ERR_BAD_ARG, "set_params cannot change the image size");
    // K1a reads the views through the staging built at upload (zero borders sized for the upload's disparity reach, per-view column phase
    // phi = gx * min_disp mod 4, line-image pitch): it may only run again for the same pairs, the same min_disp and no further reach.
    // Other parameter sets (e.g. the full range after a disparity-slice cost volume, for SGM / WTA) are accepted, but SVA_STAGE_AD then
    // needs a new upload.
    const sva_params& u = c->up_prm;
    bool same = p->reserved[0] == u.reserved[0] && p->n_pairs == u.n_pairs && p->min_disp == u.min_disp && p->win_half == u.win_half && (p->num_disp + 31) / 32 <= (u.num_disp + 31) / 32;
    for (int i = 0; same && i < p->n_pairs; i++) same = p->pair_gx[i] == u.pair_gx[i] && p->pair_gy[i] == u.pair_gy[i];
    c->ad_params_ok = same;
    c->ad_y0 = c->ad_y1 = c->cost_y0 = c->cost_y1 = 0;
    c->prm = *p;
    c->win_y0 = 0; c->win_rows = 0;
    c->pair_begin = 0; c->pair_end = p->n_pairs;
    c->have_ad = c->have_cost = c->have_sgm = c->have_disp = false;  // volumes of the old disparity range are not valid for the new one
    return SVA_OK;
}

int sva_frame_sgm_directions(sva_ctx* c, const void* cost_dev, int32_t slice_disp, uint32_t dir_mask, int32_t rows_alloc, void** out_s_ptr, size_t* out_bytes) {
    if (!c || !cost_dev) return SVA_ERR_BAD_ARG;
    if (!c->have_frame) return c->fail(SVA_ERR_STATE, "no frame uploaded");
    SVA_CUDA_OK(c, cudaSetDevice(c->device));
    SVA_TRY(sva_run_sgm_dirs(c, (const uint16_t*)cost_dev, slice_disp, dir_mask, rows_alloc));
    const int rows = rows_alloc > c->prm.height ? rows_alloc : c->prm.height;
    if (out_s_ptr) *out_s_ptr = c->S.p;
    if (out_bytes) *out_bytes = (size_t)c->prm.width * rows * c->prm.num_disp * 2;
    return SVA_OK;
}

int sva_frame_rows_begin(sva_ctx* c, int32_t y0, int32_t rows) {
    if (!c) return SVA_ERR_BAD_ARG;
    if (!c->have_frame) return c->fail(SVA_ERR_STATE, "no frame uploaded");
    const sva_params& p = c->prm;
    if (y0 < 0 || rows < 1 || y0 + rows > p.height) return c->fail(SVA_ERR_BAD_ARG, "rows_begin: bad row block");
    SVA_CUDA_OK(c, cudaSetDevice(c->device));
    const size_t row_bytes = (size_t)p.width * p.num_disp * sizeof(uint16_t);
    SVA_TRY(c->reserve(c->S, row_bytes * p.height + 64));
    SVA_CUDA_OK(c, cudaMemsetAsync((uint8_t*)c->S.p + row_bytes * y0, 0, row_bytes * rows, c->stream));
    c->s_prezeroed = false;
    c->have_sgm = false;
    c->win_y0 = y0; c->win_rows = rows == p.height ? 0 : rows;  // SVA_STAGE_AD / SVA_STAGE_BOX now compute what this block needs
    // (the volumes keep what they hold: [ad_y0, ad_y1) / [cost_y0, cost_y1) say which rows, and every consumer checks its rows against them)
    return SVA_OK;
}

int sva_frame_sgm_rows(sva_ctx* c, int32_t group, int32_t y0, int32_t rows, const void* state_in, void* state_out) {
    if (!c) return SVA_ERR_BAD_ARG;
    if (!c->have_cost) return c->fail(SVA_ERR_STATE, "sgm_rows: no cost volume");
    if (y0 < c->cost_y0 || y0 + rows > c->cost_y1) return c->fail(SVA_ERR_STATE, "sgm_rows: the cost volume was not computed for these rows");
    SVA_CUDA_OK(c, cudaSetDevice(c->device));
    SVA_TRY(sva_run_sgm_rows(c, group, y0, rows, (const uint16_t*)state_in, (uint16_t*)state_out));
    c->have_sgm = true;
    return SVA_OK;
}

int sva_frame_wta_rows(sva_ctx* c, const void* s_rows_dev, int32_t y0, int32_t rows) {
    if (!c) return SVA_ERR_BAD_ARG;
    if (!c->have_frame) return c->fail(SVA_ERR_STATE, "no frame uploaded");
    SVA_CUDA_OK(c, cudaSetDevice(c->device));
    if (!s_rows_dev) {  // the context's own aggregation volume
        if (!c->S.p || y0 < 0 || rows < 1 || y0 + rows > c->prm.height) return c->fail(SVA_ERR_BAD_ARG, "wta_rows: bad row block");
        s_rows_dev = c->S.as<uint16_t>() + (size_t)y0 * c->prm.width * c->prm.num_disp;
    }
    SVA_TRY(sva_run_wta_rows(c, (const uint16_t*)s_rows_dev, y0, rows));
    c->have_disp = true;
    return SVA_OK;
}

int sva_frame_download_disparity_rows(sva_ctx* c, int32_t rows, uint16_t* out_disp, float* out_sub) {
    if (!c || !out_disp || rows < 1 || rows > c->prm.height) return SVA_ERR_BAD_ARG;
    if (!c->have_disp) return c->fail(SVA_ERR_STATE, "disparity not computed");
    SVA_CUDA_OK(c, cudaSetDevice(c->device));
    const size_t px = (size_t)c->prm.width * rows;
    SVA_CUDA_OK(c, cudaMemcpyAsync(out_disp, c->disp.p, px * 2, cudaMemcpyDeviceToHost, c->stream));
    if (out_sub) SVA_CUDA_OK(c, cudaMemcpyAsync(out_sub, c->subpix.p, px * 4, cudaMemcpyDeviceToHost, c->stream));
    SVA_CUDA_OK(c, cudaStreamSynchronize(c->stream));
    return SVA_OK;
}

}  // extern "C"

/* ---- streaming form of sva_depth_from_array: a capture stream, two frames in flight ---------------------------------------------
 * submit(t) uploads frame t on a copy stream, runs the stages on the compute stream and downloads the maps on a second copy stream;
 * it returns at once.  Frame t+1's upload overlaps frame t's compute and frame t-1's download (two IoSets, swapped per frame).
 * The host buffers (inputs and outputs) must stay valid until sva_stream_wait(ticket) returns; pin them for real overlap. */
void sva_swap_io(sva_ctx* c) {
    c->io_swapped = !c->io_swapped;
    std::swap(c->pad_ref, c->alt.pad_ref); std::swap(c->pad_imgs, c->alt.pad_imgs); std::swap(c->ref_img, c->alt.ref_img);
    std::swap(c->other_imgs, c->alt.other_imgs); std::swap(c->lines, c->alt.lines); std::swap(c->mask, c->alt.mask);
    std::swap(c->disp, c->alt.disp); std::swap(c->subpix, c->alt.subpix); std::swap(c->ad2_zero_key, c->alt.ad2_zero_key);
}

int sva_stream_open(sva_ctx* c) {
    if (c->h2d_stream) return SVA_OK;
    SVA_CUDA_OK(c, cudaStreamCreateWithFlags(&c->h2d_stream, cudaStreamNonBlocking));
    SVA_CUDA_OK(c, cudaStreamCreateWithFlags(&c->d2h_stream, cudaStreamNonBlocking));
    SVA_CUDA_OK(c, cudaEventCreate(&c->ev_mark));
    for (int i = 0; i < 2; i++) {
        SVA_CUDA_OK(c, cudaEventCreateWithFlags(&c->ev_h2d[i], cudaEventDisableTiming));
        SVA_CUDA_OK(c, cudaEventCreateWithFlags(&c->ev_compute[i], cudaEventDisableTiming));
        SVA_CUDA_OK(c, cudaEventCreate(&c->ev_done[i]));
    }
    return SVA_OK;
}

// wait for every frame in flight on the capture stream (their tickets stay waitable: their events have completed)
int sva_stream_drain(sva_ctx* c) {
    SVA_CUDA_OK(c, cudaStreamSynchronize(c->h2d_stream));
    if (c->ad_stream) SVA_CUDA_OK(c, cudaStreamSynchronize(c->ad_stream));
    SVA_CUDA_OK(c, cudaStreamSynchronize(c->stream));
    SVA_CUDA_OK(c, cudaStreamSynchronize(c->d2h_stream));
    c->ev_box_valid = false;
    return SVA_OK;
}

// The capture-stream pipeline behind sva_stream_submit, for a checked frame whose geometry matches the frames in flight (or with none in
// flight).  view_kind says where the views live (stage_frame); sva_depth_groups runs its groups through here with the views in its stack.
// out_disp may be NULL only here, not in sva_stream_submit: the maps are then not downloaded (see below).
int sva_stream_enqueue(sva_ctx* c, const sva_params* p, const sva_image_u8* ref, const sva_image_u8* others, const sva_image_u8* mask,
                       cudaMemcpyKind view_kind, uint16_t* out_disp, float* out_subpix, int64_t* out_ticket) {
    const int64_t t = c->stream_ticket;
    const int slot = (int)(t & 1);
    if (t >= 2) SVA_CUDA_OK(c, cudaEventSynchronize(c->ev_done[slot]));  // frame t-2 is out: its IoSet is free again
    sva_swap_io(c);
    cudaStream_t compute = c->stream;
    c->stream = c->h2d_stream;
    int rc = stage_frame(c, p, ref, others, mask, view_kind);
    c->stream = compute;
    if (rc != SVA_OK) { sva_swap_io(c); return rc; }  // (allocation failure): back onto the IoSet of frame t-1, the ticket is not consumed
    SVA_CUDA_OK(c, cudaEventRecord(c->ev_h2d[slot], c->h2d_stream));
    // (only where the SGM launches are not paced — c1-sized rows: next to paced launches the intruder costs more than it hides: c2 e2e 1.67 -> 1.76 ms)
    if (c->tune_stream_ad_ahead && c->win_rows == 0 && (c->tune_stream_ad_ahead > 1 || (size_t)p->width * p->num_disp * 4 < 768 * 1024)) {
        // K1a of this frame depends on nothing but its upload, and the AD volume is free as soon as the previous frame's K1b has read it: run
        // it on a stream of its own, so that it executes NEXT TO the previous frame's first SGM launches (single horizontal directions: H warps
        // bound by HBM latency, the SMs mostly idle) instead of after its K3.  K1b and everything after it stay in order on the compute stream.
        if (!c->ad_stream) {
            SVA_CUDA_OK(c, cudaStreamCreateWithFlags(&c->ad_stream, cudaStreamNonBlocking));
            SVA_CUDA_OK(c, cudaEventCreateWithFlags(&c->ev_ad, cudaEventDisableTiming));
            SVA_CUDA_OK(c, cudaEventCreateWithFlags(&c->ev_box, cudaEventDisableTiming));
            c->ev_box_valid = false;
        }
        SVA_CUDA_OK(c, cudaStreamWaitEvent(c->ad_stream, c->ev_h2d[slot], 0));
        if (c->ev_box_valid) SVA_CUDA_OK(c, cudaStreamWaitEvent(c->ad_stream, c->ev_box, 0));
        else {  // first frame of the stream (or after a drain): whatever the compute stream still does with AP comes first
            SVA_CUDA_OK(c, cudaEventRecord(c->ev_box, compute));
            SVA_CUDA_OK(c, cudaStreamWaitEvent(c->ad_stream, c->ev_box, 0));
        }
        c->in_stream_submit = true;
        c->stream = c->ad_stream;
        rc = run_stage(c, SVA_STAGE_AD);
        c->stream = compute;
        if (rc == SVA_OK) rc = cudaEventRecord(c->ev_ad, c->ad_stream) == cudaSuccess && cudaStreamWaitEvent(compute, c->ev_ad, 0) == cudaSuccess ? SVA_OK : SVA_ERR_CUDA;
        if (rc == SVA_OK) rc = run_stage(c, SVA_STAGE_BOX);
        if (rc == SVA_OK) {
            rc = cudaEventRecord(c->ev_box, compute) == cudaSuccess ? SVA_OK : SVA_ERR_CUDA;
            c->ev_box_valid = rc == SVA_OK;
        }
        if (rc == SVA_OK) rc = run_stage(c, SVA_STAGE_SGM);
        c->in_stream_submit = false;
        SVA_TRY(rc);
    } else {
        SVA_CUDA_OK(c, cudaStreamWaitEvent(compute, c->ev_h2d[slot], 0));
        SVA_TRY(run_stage(c, SVA_STAGE_ALL));
    }
    SVA_CUDA_OK(c, cudaEventRecord(c->ev_compute[slot], compute));
    SVA_CUDA_OK(c, cudaStreamWaitEvent(c->d2h_stream, c->ev_compute[slot], 0));
    const size_t px = (size_t)p->width * p->height;
    // out_disp == NULL (sva_depth_groups_fused): no download.  The maps stay in this frame's IoSet; work the caller enqueues on the compute
    // stream after this call reads them before K3 of frame t + 2, the next writer of that IoSet's maps.
    if (out_disp) SVA_CUDA_OK(c, cudaMemcpyAsync(out_disp, c->disp.p, px * 2, cudaMemcpyDeviceToHost, c->d2h_stream));
    if (out_disp && out_subpix) SVA_CUDA_OK(c, cudaMemcpyAsync(out_subpix, c->subpix.p, px * 4, cudaMemcpyDeviceToHost, c->d2h_stream));
    SVA_CUDA_OK(c, cudaEventRecord(c->ev_done[slot], c->d2h_stream));
    c->stream_ticket = t + 1;
    *out_ticket = t;
    return SVA_OK;
}

extern "C" {

int sva_stream_submit(sva_ctx* c, const sva_params* p, const sva_image_u8* ref, const sva_image_u8* others, const sva_image_u8* mask,
                      uint16_t* out_disp, float* out_subpix, int64_t* out_ticket) {
    if (!c || !out_disp || !out_ticket) return SVA_ERR_BAD_ARG;
    SVA_CUDA_OK(c, cudaSetDevice(c->device));
    SVA_TRY(sva_stream_open(c));
    if (c->stream_ticket > 0 && p && (p->width != c->prm.width || p->height != c->prm.height || p->num_disp != c->prm.num_disp || p->n_pairs != c->prm.n_pairs ||
                       p->win_half != c->prm.win_half || p->min_disp != c->prm.min_disp || p->reserved[0] != c->prm.reserved[0])) {
        SVA_TRY(sva_stream_drain(c));  // a different geometry re-allocates workspaces: no frame in flight may still use the old ones
    }
    SVA_TRY(check_frame_args(c, p, ref, others, mask));  // a bad frame must not disturb the frames in flight: nothing is touched before this
    return sva_stream_enqueue(c, p, ref, others, mask, cudaMemcpyHostToDevice, out_disp, out_subpix, out_ticket);
}

int sva_stream_wait(sva_ctx* c, int64_t ticket) {
    if (!c || !c->h2d_stream) return SVA_ERR_BAD_ARG;
    if (ticket < 0 || ticket >= c->stream_ticket) return c->fail(SVA_ERR_BAD_ARG, "unknown ticket");
    if (ticket + 2 < c->stream_ticket) return SVA_OK;  // retired when its slot was reused
    SVA_CUDA_OK(c, cudaSetDevice(c->device));
    SVA_CUDA_OK(c, cudaEventSynchronize(c->ev_done[ticket & 1]));
    return SVA_OK;
}

/* device-clock stopwatch of the streaming path: mark() stamps the upload stream, elapsed(ticket) is the time from the mark to the end of
 * that frame's download (ticket must be one of the two most recent) */
int sva_stream_mark(sva_ctx* c) {
    if (!c) return SVA_ERR_BAD_ARG;
    SVA_CUDA_OK(c, cudaSetDevice(c->device));
    SVA_TRY(sva_stream_open(c));
    SVA_CUDA_OK(c, cudaStreamSynchronize(c->stream));
    SVA_CUDA_OK(c, cudaStreamSynchronize(c->d2h_stream));
    SVA_CUDA_OK(c, cudaEventRecord(c->ev_mark, c->h2d_stream));
    return SVA_OK;
}
int sva_stream_elapsed(sva_ctx* c, int64_t ticket, float* out_ms) {
    if (!c || !out_ms || !c->h2d_stream) return SVA_ERR_BAD_ARG;
    if (ticket < 0 || ticket >= c->stream_ticket || ticket + 2 < c->stream_ticket) return c->fail(SVA_ERR_BAD_ARG, "ticket is not one of the two most recent");
    SVA_CUDA_OK(c, cudaEventSynchronize(c->ev_done[ticket & 1]));
    SVA_CUDA_OK(c, cudaEventElapsedTime(out_ms, c->ev_mark, c->ev_done[ticket & 1]));
    return SVA_OK;
}

}  // extern "C"
