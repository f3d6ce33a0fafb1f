// sva_groups.cu — sva_depth_groups: the depth map of every reference view of ONE array frame in one call (getGroups, SURVEY §8 f3).
//
// The frame's cameras are uploaded once into a device stack (tight W x H views, camera i at cam_stack + i * W * H) on a copy stream of
// their own, in order of first use, with one event per camera.  The groups then run through the capture-stream pipeline of
// sva_stream_submit (sva_api.cu: two IoSets, K1a of group g + 1 next to group g's SGM, the maps of group g downloaded straight into the
// caller's buffers while later groups compute), each staging its views device to device from the stack once its own cameras are in.  In
// census mode every camera's signatures are computed once, into a second stack that K1a reads directly: 25 transforms for the 13 CHESS
// groups of a 5 x 5 frame instead of 55.
//
// sva_depth_groups_fused runs the same pipeline without the per-group downloads: each group's maps are splatted into the fusion's planes
// (k_fuse.cu) on the compute stream right after its K3, and the fused maps are the only download.
#include <vector>

#include "sva_common.cuh"

int check_params(sva_ctx* c, const sva_params* p);
int sva_stream_open(sva_ctx* c);
int sva_stream_drain(sva_ctx* c);
void sva_swap_io(sva_ctx* c);
int sva_stream_enqueue(sva_ctx* c, const sva_params* p, const sva_image_u8* ref, const sva_image_u8* others, const sva_image_u8* mask,
                       cudaMemcpyKind view_kind, uint16_t* out_disp, float* out_subpix, int64_t* out_ticket);
int sva_census_stack(sva_ctx* ctx, const uint8_t* stack, int W, int H, const int* cams, int n, uint64_t* sig, cudaStream_t stream);
int sva_fuse_check(sva_ctx* c, int W, int H, int grid_cols, int n_cameras, const int32_t* refs, int n_views, int target, const sva_fuse_params* f,
                   const sva_image_u8* mask);
int sva_fuse_begin(sva_ctx* c, int W, int H, int G, bool has_mask);
int sva_fuse_splat(sva_ctx* c, int W, int H, const uint16_t* disp, const float* sub, size_t view_stride, int v0, int n, const int* gx, const int* gy);
int sva_fuse_finish(sva_ctx* c, int W, int H, int G, const sva_fuse_params* f, const sva_image_u8* mask, uint16_t* out_disp, float* out_sub,
                    uint8_t* out_support);

// group g's parameters: the template with the grid offsets of its pairs, gx = col(other) - col(ref), gy = row(other) - row(ref)
static void group_params(const sva_params& tpl, const int32_t* pairs, int n, int grid_cols, sva_params& out) {
    out = tpl;
    out.n_pairs = n;
    for (int j = 0; j < n; j++) {
        const int ref = pairs[2 * j], other = pairs[2 * j + 1];
        out.pair_gx[j] = other % grid_cols - ref % grid_cols;
        out.pair_gy[j] = other / grid_cols - ref / grid_cols;
    }
}

static int check_view(sva_ctx* c, const sva_image_u8& im, int W, int H, const char* what, int index) {
    if (im.cols != W || im.rows != H || im.step < (size_t)W)
        return c->fail(SVA_ERR_BAD_ARG, std::string("depth_groups: ") + what + " " + std::to_string(index) + " is not width x height");
    return SVA_OK;
}

// Every refusal of sva_depth_groups but those of its outputs, before anything is enqueued.  first[g] = index of group g's first pair.
static int check_groups(sva_ctx* c, const sva_params* p, int32_t grid_cols, const sva_image_u8* images, int32_t n_images, const int32_t* pairs,
                        const int32_t* sizes, int32_t n_groups, int32_t b, int32_t e, const sva_image_u8* masks, std::vector<int64_t>& first) {
    if (!p) return c->fail(SVA_ERR_BAD_ARG, "depth_groups: null params");
    if (n_groups < 0 || (n_groups > 0 && (!pairs || !sizes))) return c->fail(SVA_ERR_BAD_ARG, "depth_groups: null pairs / sizes");
    if (b < 0 || e > n_groups || b > e) return c->fail(SVA_ERR_BAD_ARG, "depth_groups: group range outside [0, n_groups]");
    if (grid_cols < 1 || n_images < 1 || n_images % grid_cols) return c->fail(SVA_ERR_BAD_ARG, "depth_groups: n_images must be a positive multiple of grid_cols");
    if (!images) return c->fail(SVA_ERR_BAD_ARG, "depth_groups: null images");
    bool tpl_ok = p->n_pairs == 0;
    for (int i = 0; i < SVA_MAX_PAIRS; i++) tpl_ok = tpl_ok && p->pair_gx[i] == 0 && p->pair_gy[i] == 0;
    if (!tpl_ok) return c->fail(SVA_ERR_BAD_ARG, "depth_groups: the template's n_pairs, pair_gx and pair_gy must be zero (each group's come from its pairs)");
    first.assign(n_groups + 1, 0);
    for (int g = 0; g < n_groups; g++) {
        if (sizes[g] < 0) return c->fail(SVA_ERR_BAD_ARG, "depth_groups: negative group size");
        first[g + 1] = first[g] + sizes[g];
    }
    for (int g = 0; g < n_groups; g++) {
        const int32_t* pr = pairs + 2 * first[g];
        for (int j = 0; j < sizes[g]; j++) {
            const int ref = pr[2 * j], other = pr[2 * j + 1];
            if (ref < 0 || ref >= n_images || other < 0 || other >= n_images)
                return c->fail(SVA_ERR_BAD_ARG, "depth_groups: group " + std::to_string(g) + " names a camera outside [0, n_images)");
            if (ref != pr[0]) return c->fail(SVA_ERR_BAD_ARG, "depth_groups: the pairs of group " + std::to_string(g) + " do not share one reference");
            if (other == ref) return c->fail(SVA_ERR_BAD_ARG, "depth_groups: group " + std::to_string(g) + " pairs a camera with itself");
        }
        if (sizes[g] > SVA_MAX_PAIRS) return c->fail(SVA_ERR_BAD_ARG, "depth_groups: group " + std::to_string(g) + " has more than 32 pairs");
        sva_params gp;
        group_params(*p, pr, sizes[g], grid_cols, gp);
        const int rc = check_params(c, &gp);
        if (rc != SVA_OK) return c->fail(rc, "depth_groups: group " + std::to_string(g) + ": " + c->err);
    }
    const int W = p->width, H = p->height;
    for (int g = b; g < e; g++) {
        const int32_t* pr = pairs + 2 * first[g];
        for (int j = 0; j < 2 * sizes[g]; j++) {
            const sva_image_u8& im = images[pr[j]];
            if (!im.data) return c->fail(SVA_ERR_BAD_ARG, "depth_groups: camera " + std::to_string(pr[j]) + " is read by group " + std::to_string(g) + " but has no data");
            SVA_TRY(check_view(c, im, W, H, "camera", pr[j]));
        }
        if (masks && masks[g - b].data) SVA_TRY(check_view(c, masks[g - b], W, H, "mask of group", g));
    }
    return SVA_OK;
}

// sva_depth_groups_fused: the target and outputs of the fusion the groups' maps go into instead of the caller's buffers
struct GroupsFusion {
    int target;
    const sva_fuse_params* f;
    const sva_image_u8* mask;
    uint16_t* out_disp;
    float* out_subpix;
    uint8_t* out_support;
};

// The groups [group_begin, group_end) of a checked call, their maps into out_disp / out_subpix or, with fuse, into the fusion.
static int run_groups(sva_ctx* c, const sva_params* p, int32_t grid_cols, const sva_image_u8* images, int32_t n_images, const int32_t* pairs,
                      const int32_t* sizes, const std::vector<int64_t>& first, int32_t group_begin, int32_t group_end, const sva_image_u8* masks,
                      uint16_t* const* out_disp, float* const* out_subpix, const GroupsFusion* fuse) {
    SVA_CUDA_OK(c, cudaSetDevice(c->device));
    const int W = p->width, H = p->height;
    const size_t px = (size_t)W * H;
    const bool census = p->reserved[0] == SVA_COST_CENSUS;
    SVA_TRY(sva_stream_open(c));
    // Capture-stream frames still in flight complete first (their tickets stay waitable).  With both IoSets idle, group g of a call then
    // always stages into the same one of the two, so a second call of the same geometry and groups finds every buffer already sized.
    SVA_TRY(sva_stream_drain(c));
    if (c->io_swapped) sva_swap_io(c);
    if (!c->stack_stream) SVA_CUDA_OK(c, cudaStreamCreateWithFlags(&c->stack_stream, cudaStreamNonBlocking));
    while ((int)c->ev_cam.size() < n_images) {
        cudaEvent_t ev;
        SVA_CUDA_OK(c, cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
        c->ev_cam.push_back(ev);
    }
    {
        cudaStream_t compute = c->stream;
        c->stream = c->stack_stream;  // a (guarded) allocation initialises its bytes on the stream that then writes the stack
        int rc = c->reserve(c->cam_stack, px * n_images);
        if (rc == SVA_OK && census) rc = c->reserve(c->cam_sig, px * sizeof(uint64_t) * n_images);
        c->stream = compute;
        SVA_TRY(rc);
    }
    if (fuse) SVA_TRY(sva_fuse_begin(c, W, H, group_end - group_begin, fuse->mask != nullptr));  // on the compute stream, before the first splat
    uint8_t* stack = c->cam_stack.as<uint8_t>();
    // upload every camera once, in order of first use; census: its signatures too
    std::vector<char> in_stack(n_images, 0);
    for (int g = group_begin; g < group_end; g++) {
        const int32_t* pr = pairs + 2 * first[g];
        int fresh[SVA_MAX_PAIRS + 1], n_fresh = 0;
        for (int j = 0; j < 2 * sizes[g]; j++) {
            const int cam = pr[j];
            if (in_stack[cam]) continue;
            in_stack[cam] = 1;
            fresh[n_fresh++] = cam;
            SVA_CUDA_OK(c, cudaMemcpy2DAsync(stack + px * cam, W, images[cam].data, images[cam].step, W, H, cudaMemcpyHostToDevice, c->stack_stream));
        }
        if (census) SVA_TRY(sva_census_stack(c, stack, W, H, fresh, n_fresh, c->cam_sig.as<uint64_t>(), c->stack_stream));
        for (int i = 0; i < n_fresh; i++) SVA_CUDA_OK(c, cudaEventRecord(c->ev_cam[fresh[i]], c->stack_stream));
    }
    // the groups through the capture-stream pipeline, views staged from the stack
    int rc = SVA_OK;
    for (int g = group_begin; g < group_end && rc == SVA_OK; g++) {
        const int32_t* pr = pairs + 2 * first[g];
        const int n = sizes[g], ref = pr[0];
        sva_params gp;
        group_params(*p, pr, n, grid_cols, gp);
        const sva_image_u8 rv{stack + px * ref, H, W, (size_t)W};
        sva_image_u8 ov[SVA_MAX_PAIRS];
        for (int j = 0; j < n; j++) ov[j] = sva_image_u8{stack + px * pr[2 * j + 1], H, W, (size_t)W};
        for (int j = 0; j < 2 * n && rc == SVA_OK; j++)
            if (cudaStreamWaitEvent(c->h2d_stream, c->ev_cam[pr[j]], 0) != cudaSuccess) rc = c->fail(SVA_ERR_CUDA, "depth_groups: cudaStreamWaitEvent");
        if (rc != SVA_OK) break;
        if (census) {
            c->sig_stack = c->cam_sig.as<uint64_t>();
            c->sig_ref = ref;
            for (int j = 0; j < n; j++) c->sig_view[j] = pr[2 * j + 1];
        }
        const sva_image_u8* mask = masks && masks[g - group_begin].data ? &masks[g - group_begin] : nullptr;
        int64_t ticket = 0;
        if (fuse) {
            // no download: the group's maps go from its IoSet into the fusion's planes on the compute stream, right after its K3
            rc = sva_stream_enqueue(c, &gp, &rv, ov, mask, cudaMemcpyDeviceToDevice, nullptr, nullptr, &ticket);
            const int gx = fuse->target % grid_cols - ref % grid_cols, gy = fuse->target / grid_cols - ref / grid_cols;
            if (rc == SVA_OK)
                rc = sva_fuse_splat(c, W, H, c->disp.as<uint16_t>(), p->subpixel == 1 ? c->subpix.as<float>() : nullptr, 0, g - group_begin, 1, &gx, &gy);
        } else {
            rc = sva_stream_enqueue(c, &gp, &rv, ov, mask, cudaMemcpyDeviceToDevice, out_disp[g - group_begin], out_subpix ? out_subpix[g - group_begin] : nullptr, &ticket);
        }
        c->sig_stack = nullptr;
    }
    if (rc == SVA_OK && fuse)
        rc = sva_fuse_finish(c, W, H, group_end - group_begin, fuse->f, fuse->mask, fuse->out_disp, fuse->out_subpix, fuse->out_support);
    // synchronous: every map is in the caller's buffers, and nothing reads the stack any more, when this returns (also after a failure)
    const std::string err = c->err;
    const int rc_drain = sva_stream_drain(c);
    const int rc_stack = cudaStreamSynchronize(c->stack_stream) == cudaSuccess ? SVA_OK : c->fail(SVA_ERR_CUDA, "depth_groups: cudaStreamSynchronize");
    if (rc != SVA_OK) { c->err = err; return rc; }
    return rc_drain != SVA_OK ? rc_drain : rc_stack;
}

extern "C" int sva_depth_groups(sva_ctx* c, const sva_params* p, int32_t grid_cols, const sva_image_u8* images, int32_t n_images, const int32_t* pairs,
                                const int32_t* sizes, int32_t n_groups, int32_t group_begin, int32_t group_end, const sva_image_u8* masks,
                                uint16_t* const* out_disp, float* const* out_subpix) {
    if (!c) return SVA_ERR_BAD_ARG;
    std::vector<int64_t> first;
    SVA_TRY(check_groups(c, p, grid_cols, images, n_images, pairs, sizes, n_groups, group_begin, group_end, masks, first));
    if (group_end > group_begin && !out_disp) return c->fail(SVA_ERR_BAD_ARG, "depth_groups: null out_disp");
    for (int g = group_begin; g < group_end; g++)
        if (!out_disp[g - group_begin]) return c->fail(SVA_ERR_BAD_ARG, "depth_groups: null out_disp of group " + std::to_string(g));
    if (group_begin == group_end) return SVA_OK;
    return run_groups(c, p, grid_cols, images, n_images, pairs, sizes, first, group_begin, group_end, masks, out_disp, out_subpix, nullptr);
}

extern "C" int sva_depth_groups_fused(sva_ctx* c, const sva_params* p, int32_t grid_cols, const sva_image_u8* images, int32_t n_images,
                                      const int32_t* pairs, const int32_t* sizes, int32_t n_groups, const sva_image_u8* masks, int32_t target,
                                      const sva_fuse_params* f, const sva_image_u8* target_mask, uint16_t* out_disp, float* out_subpix,
                                      uint8_t* out_support) {
    if (!c) return SVA_ERR_BAD_ARG;
    std::vector<int64_t> first;
    SVA_TRY(check_groups(c, p, grid_cols, images, n_images, pairs, sizes, n_groups, 0, n_groups, masks, first));
    // the views are the groups, each with its reference camera (check_groups has made sure every group has one, inside [0, n_images))
    std::vector<int32_t> refs(n_groups);
    for (int g = 0; g < n_groups; g++) refs[g] = pairs[2 * first[g]];
    SVA_TRY(sva_fuse_check(c, p->width, p->height, grid_cols, n_images, refs.data(), n_groups, target, f, target_mask));
    if (!out_disp) return c->fail(SVA_ERR_BAD_ARG, "depth_groups_fused: null out_disp");
    const GroupsFusion fuse{target, f, target_mask, out_disp, out_subpix, out_support};
    return run_groups(c, p, grid_cols, images, n_images, pairs, sizes, first, 0, n_groups, masks, nullptr, nullptr, &fuse);
}
