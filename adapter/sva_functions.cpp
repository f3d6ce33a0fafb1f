// adapter/sva_functions.cpp — the reference-side binding: the hot functions of include/functions.h and Camera.h of
// Nahuel-M/StereoVisionArray re-implemented as thin calls into libsva_b200.so (include/sva_c_api.h).
//
// Integration (INTEGRATION.md): add this file to the reference's build INSTEAD of the bodies it replaces in
// src/functions.cpp / src/Camera.cpp, add include/ of this repo to the include path and link libsva_b200.so.  The signatures
// are the reference's own (functions.h:22,26,34-38,45; Camera.h:12-13), so src/CameraStereoVision.cpp and the dlibFaceSelect
// ROI path call them unchanged.  It compiles against real OpenCV (cv::Mat) — and, for this repo's tests, against the minimal
// stand-in in oracle/cvshim.  No reference source is copied: the headers are the reference tree's own, or for this repo's tests
// the stand-in declarations in adapter/refshim where no reference tree is given.
//
// Error behaviour: the reference surfaces failures as cv::Exception; a non-zero sva status is turned back into one.
// Ownership: every function returns a freshly allocated Mat / vector, inputs are not mutated, no pointer is retained.
#include <array>
#include <string>
#include <vector>

#include "Camera.h"
#include "functions.h"
#include "dlibFaceSelect.h"
#include "sva_c_api.h"
#include "sva_rows_stream.h"

namespace {

int g_device = 0;  // svaSelectDevice: one process per GPU picks its GPU before the first call
sva_ctx* ctx() {  // one context per process (the reference is single-threaded, functions.h has no handle argument)
    static sva_ctx* c = nullptr;
    if (!c) {
        int rc = sva_create(g_device, &c);
        if (rc != SVA_OK) throw cv::Exception(std::string("sva_create failed: a B200 GPU is required (status ") + std::to_string(rc) + ")");
    }
    return c;
}
void check(int rc, const char* what) {
    if (rc < 0) throw cv::Exception(std::string(what) + ": " + sva_last_error(ctx()));
}
sva_image_u8 view(const cv::Mat& m) { return sva_image_u8{m.data, m.rows, m.cols, (size_t)m.step}; }
sva_camera cam(const Camera& c) { return sva_camera{{c.pos3D.x, c.pos3D.y, c.pos3D.z}, c.f, c.pixel_size}; }

}  // namespace

// ---- Camera (include/Camera.h:6-21, src/Camera.cpp) ----
#ifndef SVA_ADAPTER_KEEP_REFERENCE_CAMERA
Camera::Camera(double focal_length, cv::Point3d position, double pixel_size) : pos3D{position}, f{focal_length}, pixel_size{pixel_size} {}
Camera::~Camera() {}
cv::Point2i Camera::project(cv::Point3d Pos3D) {
    sva_camera c = cam(*this);
    double p[3] = {Pos3D.x, Pos3D.y, Pos3D.z};
    int32_t out[2];
    sva_camera_project(&c, p, out);
    return cv::Point2i{out[0], out[1]};
}
cv::Point3d Camera::inv_project(cv::Point2i pixel) {
    sva_camera c = cam(*this);
    int32_t px[2] = {pixel.x, pixel.y};
    double r[3];
    sva_camera_inv_project(&c, px, r);
    return cv::Point3d{r[0], r[1], r[2]};
}
#endif

// ---- functions.h ----
double getAbsDiff(cv::Mat& mat1, cv::Mat& mat2) {  // functions.h:38
    sva_image_u8 a = view(mat1), b = view(mat2);
    double s = 0;
    check(sva_abs_diff_u8(ctx(), &a, &b, &s), "getAbsDiff");
    return s;
}

std::vector<cv::Point2i> bresenham(cv::Point2i point1, cv::Point2i point2) {  // functions.h:45
    int cap = 2 * (std::abs(point1.x - point2.x) + std::abs(point1.y - point2.y)) + 8;
    std::vector<int32_t> xy(2 * (size_t)cap);
    int n = sva_bresenham(point1.x, point1.y, point2.x, point2.y, xy.data(), cap);
    std::vector<cv::Point2i> pts;
    for (int i = 0; i < n; i++) pts.push_back(cv::Point2i{xy[2 * i], xy[2 * i + 1]});
    return pts;
}

std::vector<std::array<int, 2>> getCameraPairs(const std::vector<Camera>& cameras, const pairType pairs) {  // functions.h:34
    int32_t out[128];
    int n = sva_get_camera_pairs((int)cameras.size(), (int)pairs, -1, out, 64);
    std::vector<std::array<int, 2>> r;
    for (int i = 0; i < n && i < 64; i++) r.push_back({out[2 * i], out[2 * i + 1]});  // n may exceed the capacity; only 64 pairs were written
    return r;
}
std::vector<std::array<int, 2>> getCameraPairs(const std::vector<Camera>& cameras, const pairType pair, int cameraNum) {  // functions.h:36
    int32_t out[128];
    int n = sva_get_camera_pairs((int)cameras.size(), (int)pair, cameraNum, out, 64);
    std::vector<std::array<int, 2>> r;
    for (int i = 0; i < n && i < 64; i++) r.push_back({out[2 * i], out[2 * i + 1]});  // n may exceed the capacity; only 64 pairs were written
    return r;
}

cv::Mat shiftPerspectiveWithDisparity(Camera& inputCam, Camera& outputCam, cv::Mat& disparity, cv::Mat& image) {  // functions.h:26
    cv::Mat out{image.size(), image.type()};
    sva_camera ci = cam(inputCam), co = cam(outputCam);
    sva_image_u8 d = view(disparity), im = view(image);
    check(sva_shift_perspective_with_disparity(ctx(), &ci, &co, &d, &im, out.data), "shiftPerspectiveWithDisparity");
    return out;
}

cv::Mat improveWithDisparity(cv::Mat& disparity, cv::Mat centerImage, std::vector<cv::Mat>& images, std::vector<std::array<Camera, 2>>& cameras,
                             int windowSize) {  // functions.h:22; the GUI calls of src/functions.cpp:20-21,42-43 do not cross the ABI
    cv::Mat mask = getFaceMask(centerImage);  // src/functions.cpp:13 — the ROI stays the reference's own (dlibFaceSelect)
    cv::Mat out{disparity.size(), disparity.type()};
    std::vector<sva_image_u8> imgs;
    std::vector<sva_camera> cams;
    for (size_t i = 0; i < cameras.size(); i++) {
        imgs.push_back(view(images[i]));
        cams.push_back(cam(cameras[i][0]));
        cams.push_back(cam(cameras[i][1]));
    }
    sva_image_u8 d = view(disparity), c = view(centerImage), m = view(mask);
    check(sva_improve_with_disparity(ctx(), &d, &c, imgs.data(), cams.data(), (int)cameras.size(), &m, windowSize, out.data), "improveWithDisparity");
    return out;
}

// ---- the batched replacement of the loop nest in main (src/CameraStereoVision.cpp:49-95) — the one call the driver gains ----
cv::Mat svaMatchLiteral(std::vector<cv::Mat>& images, std::vector<Camera>& cameras, std::vector<std::array<int, 2>>& pairs, cv::Mat& mask, int kernelSize,
                        double rayNear, double rayFar) {
    cv::Mat out{images[pairs[0][0]].size(), CV_8UC1};
    std::vector<sva_image_u8> imgs;
    std::vector<sva_camera> cams;
    std::vector<int32_t> pr;
    for (auto& im : images) imgs.push_back(view(im));
    for (auto& c : cameras) cams.push_back(cam(c));
    for (auto& p : pairs) { pr.push_back(p[0]); pr.push_back(p[1]); }
    sva_image_u8 m = view(mask);
    check(sva_match_literal(ctx(), imgs.data(), cams.data(), (int)imgs.size(), pr.data(), (int)pairs.size(), &m, kernelSize, rayNear, rayFar, out.data), "svaMatchLiteral");
    return out;
}

// ---- consumers of the depth output (functions.h:24,28,30,32) ----
cv::Mat shiftPerspective2(Camera inputCam, Camera outputCam, cv::Mat& depthMap) {  // src/functions.cpp:79-104; depthMap is CV_64FC1, continuous rows
    cv::Mat src = depthMap.clone();  // clone() is continuous, whatever view the caller passed
    cv::Mat out(src.size(), src.type());
    sva_camera ci = cam(inputCam), co = cam(outputCam);
    check(sva_shift_perspective2(ctx(), &ci, &co, (const double*)src.data, src.rows, src.cols, (double*)out.data), "shiftPerspective2");
    return out;
}
cv::Mat Points3DToDepthMap(std::vector<cv::Point3d>& points, Camera camera, cv::Size resolution) {  // src/functions.cpp:118-133
    cv::Mat out(resolution, CV_64FC1);
    sva_camera c = cam(camera);
    static_assert(sizeof(cv::Point3d) == 3 * sizeof(double), "Point3d must be three packed doubles");
    check(sva_points3d_to_depth_map(ctx(), points.empty() ? nullptr : &points[0].x, (int64_t)points.size(), &c, resolution.width, resolution.height,
                                    (double*)out.data), "Points3DToDepthMap");
    return out;
}
std::vector<cv::Point3d> DepthMapToPoints3D(cv::Mat& depthMap, Camera camera, cv::Size resolution) {  // src/functions.cpp:135-146
    cv::Mat src = depthMap.clone();  // clone() is continuous, whatever view the caller passed
    std::vector<cv::Point3d> pts((size_t)src.rows * src.cols);
    sva_camera c = cam(camera);
    int64_t n = 0;
    check(sva_depth_map_to_points3d(ctx(), (const double*)src.data, src.rows, src.cols, &c, resolution.width, resolution.height,
                                    pts.empty() ? nullptr : &pts[0].x, (int64_t)pts.size(), &n), "DepthMapToPoints3D");
    pts.resize((size_t)n);
    return pts;
}
std::vector<std::vector<std::array<int, 2>>> getGroups(std::vector<Camera>& cameras, std::string groupType) {  // src/functions.cpp:107-116
    std::vector<int32_t> pairs(2 * 256), sizes(64);
    int ng = sva_get_groups((int32_t)cameras.size(), groupType.c_str(), pairs.data(), 256, sizes.data(), 64);
    if (ng < 0) throw cv::Exception("getGroups: bad argument");
    std::vector<std::vector<std::array<int, 2>>> groups;
    size_t o = 0;
    for (int g = 0; g < ng; g++) {
        std::vector<std::array<int, 2>> grp;
        for (int j = 0; j < sizes[g]; j++, o++) grp.push_back({pairs[2 * o], pairs[2 * o + 1]});
        groups.push_back(grp);
    }
    return groups;
}

// ---- every reference view of one array frame in one call (sva_depth_groups) ----
// groups as getGroups returns them (e.g. getGroups(cameras, "CHESS"), quirks included), images on a grid of gridCols columns; masks: null, or one
// per group (an empty Mat: no mask).  -> one u16 map (rows * cols; SVA_DISP_INVALID where rejected) per group, and the sub-pixel maps in *subpix
std::vector<std::vector<uint16_t>> svaDepthGroups(const sva_params& p, std::vector<cv::Mat>& images, const std::vector<std::vector<std::array<int, 2>>>& groups,
                                                  int gridCols, const std::vector<cv::Mat>* masks, std::vector<std::vector<float>>* subpix) {
    if (masks && masks->size() != groups.size()) throw cv::Exception("svaDepthGroups: one mask (or an empty Mat) per group");
    std::vector<sva_image_u8> ims, mk;
    for (auto& m : images) ims.push_back(m.empty() ? sva_image_u8{} : view(m));
    if (masks) for (auto& m : *masks) mk.push_back(m.empty() ? sva_image_u8{} : view(m));
    std::vector<int32_t> pairs, sizes;
    for (auto& g : groups) {
        sizes.push_back((int32_t)g.size());
        for (auto& pr : g) { pairs.push_back(pr[0]); pairs.push_back(pr[1]); }
    }
    const size_t n = groups.size(), px = (size_t)p.width * p.height;
    std::vector<std::vector<uint16_t>> disp(n, std::vector<uint16_t>(px));
    std::vector<std::vector<float>> sub(n, std::vector<float>(px));
    std::vector<uint16_t*> dp;
    std::vector<float*> sp;
    for (size_t g = 0; g < n; g++) { dp.push_back(disp[g].data()); sp.push_back(sub[g].data()); }
    check(sva_depth_groups(ctx(), &p, gridCols, ims.data(), (int32_t)ims.size(), pairs.data(), sizes.data(), (int32_t)n, 0, (int32_t)n, masks ? mk.data() : nullptr,
                           dp.data(), sp.data()), "svaDepthGroups");
    if (subpix) *subpix = std::move(sub);
    return disp;
}

// ---- multi-view depth fusion (sva_fuse_maps, sva_depth_groups_fused; DESIGN §3 item 6; no reference counterpart) ----
// The maps of views whose reference cameras are viewRefs (e.g. svaDepthGroups' outputs with each group's reference camera) fused into camera
// target's view on a grid of gridCols columns and nCameras cameras; subpix: null (fuse the integer maps) or one per view; targetMask: null or
// an empty Mat (no mask), or width x height.  -> the fused u16 map (SVA_DISP_INVALID where rejected); the sub-pixel map in *outSubpix and the
// number of agreeing views per pixel in *outSupport when given.
std::vector<uint16_t> svaFuseMaps(int width, int height, int gridCols, int nCameras, const std::vector<int>& viewRefs,
                                  const std::vector<std::vector<uint16_t>>& disp, const std::vector<std::vector<float>>* subpix, int target,
                                  const sva_fuse_params& f, const cv::Mat* targetMask, std::vector<float>* outSubpix, std::vector<uint8_t>* outSupport) {
    const size_t px = (size_t)width * height;
    if (viewRefs.size() != disp.size() || (subpix && subpix->size() != disp.size())) throw cv::Exception("svaFuseMaps: one reference (and map) per view");
    std::vector<const uint16_t*> dp;
    std::vector<const float*> sp;
    for (size_t g = 0; g < disp.size(); g++) {
        if (disp[g].size() != px || (subpix && (*subpix)[g].size() != px)) throw cv::Exception("svaFuseMaps: a map is not width x height");
        dp.push_back(disp[g].data());
        if (subpix) sp.push_back((*subpix)[g].data());
    }
    std::vector<int32_t> refs(viewRefs.begin(), viewRefs.end());
    std::vector<uint16_t> out(px);
    std::vector<float> sub(px);
    std::vector<uint8_t> sup(px);
    const bool masked = targetMask && !targetMask->empty();
    const sva_image_u8 mk = masked ? view(*targetMask) : sva_image_u8{};
    check(sva_fuse_maps(ctx(), width, height, gridCols, nCameras, refs.data(), (int32_t)refs.size(), dp.data(), subpix ? sp.data() : nullptr, target, &f,
                        masked ? &mk : nullptr, out.data(), sub.data(), sup.data()), "svaFuseMaps");
    if (outSubpix) *outSubpix = std::move(sub);
    if (outSupport) *outSupport = std::move(sup);
    return out;
}

// Every group of one array frame (as svaDepthGroups computes them), fused into camera target's view in one call: the group maps never leave
// the GPU.  The sub-pixel maps are fused iff p.subpixel == 1.  Equal to svaDepthGroups followed by svaFuseMaps with each group's reference.
std::vector<uint16_t> svaDepthGroupsFused(const sva_params& p, std::vector<cv::Mat>& images, const std::vector<std::vector<std::array<int, 2>>>& groups,
                                          int gridCols, int target, const sva_fuse_params& f, std::vector<float>* subpix, std::vector<uint8_t>* support,
                                          const std::vector<cv::Mat>* masks, const cv::Mat* targetMask) {
    if (masks && masks->size() != groups.size()) throw cv::Exception("svaDepthGroupsFused: one mask (or an empty Mat) per group");
    std::vector<sva_image_u8> ims, mk;
    for (auto& m : images) ims.push_back(m.empty() ? sva_image_u8{} : view(m));
    if (masks) for (auto& m : *masks) mk.push_back(m.empty() ? sva_image_u8{} : view(m));
    std::vector<int32_t> pairs, sizes;
    for (auto& g : groups) {
        sizes.push_back((int32_t)g.size());
        for (auto& pr : g) { pairs.push_back(pr[0]); pairs.push_back(pr[1]); }
    }
    const size_t px = (size_t)p.width * p.height;
    std::vector<uint16_t> out(px);
    std::vector<float> sub(px);
    std::vector<uint8_t> sup(px);
    const bool masked = targetMask && !targetMask->empty();
    const sva_image_u8 tm = masked ? view(*targetMask) : sva_image_u8{};
    check(sva_depth_groups_fused(ctx(), &p, gridCols, ims.data(), (int32_t)ims.size(), pairs.data(), sizes.data(), (int32_t)groups.size(),
                                 masks ? mk.data() : nullptr, target, &f, masked ? &tm : nullptr, out.data(), sub.data(), sup.data()),
          "svaDepthGroupsFused");
    if (subpix) *subpix = std::move(sub);
    if (support) *support = std::move(sup);
    return out;
}

// ---- one frame over several GPUs (one process per GPU; any launcher — mpirun, torchrun, a shell loop — provides rank and world) ----
// No reference counterpart (the reference is one thread): the sharding units are its pair loop (src/CameraStereoVision.cpp:55) and its
// pixel-row loop (:49).  Rank 0 calls svaCommUniqueId() and hands the 128 bytes to the others by whatever channel the launcher offers;
// every rank then calls svaCommInit (collective).  Volume-mode parameters are the C ABI's sva_params (DESIGN.md §3).
void svaSelectDevice(int device) { g_device = device; }
std::array<uint8_t, SVA_COMM_ID_BYTES> svaCommUniqueId() {
    std::array<uint8_t, SVA_COMM_ID_BYTES> id{};
    if (sva_comm_get_unique_id(id.data()) != SVA_OK) throw cv::Exception("svaCommUniqueId: libnccl.so.2 could not be loaded");
    return id;
}
void svaCommInit(const std::array<uint8_t, SVA_COMM_ID_BYTES>& id, int rank, int world) { check(sva_comm_init(ctx(), id.data(), rank, world), "svaCommInit"); }
// camera pairs sharded over the ranks, packed NCCL reduce of the AD volume onto `root` (north_star's scheme): the u16 disparity map
// (rows * cols; SVA_DISP_INVALID where rejected) on root, empty elsewhere
std::vector<uint16_t> svaDepthPairSharded(const sva_params& p, cv::Mat& ref, std::vector<cv::Mat>& others, cv::Mat* mask, int root, std::vector<float>* subpix) {
    std::vector<sva_image_u8> o;
    for (auto& m : others) o.push_back(view(m));
    sva_image_u8 r = view(ref), mk = mask ? view(*mask) : sva_image_u8{};
    std::vector<uint16_t> disp((size_t)p.width * p.height);
    std::vector<float> sub((size_t)p.width * p.height);
    check(sva_depth_pair_sharded(ctx(), &p, &r, o.data(), mask ? &mk : nullptr, root, disp.data(), sub.data()), "svaDepthPairSharded");
    if (subpix) *subpix = sub;
    return disp;
}
// image rows sharded over the ranks, path-line state handed from GPU to GPU by peer-direct stores (sva_rows_*): this rank's rows
// [y0, y0 + rows) of the map.  The first call for a geometry opens and connects the link (collective).
std::vector<uint16_t> svaDepthRowsSharded(const sva_params& p, cv::Mat& ref, std::vector<cv::Mat>& others, cv::Mat* mask, int rank, int world, int* y0, int* rows,
                                          std::vector<float>* subpix) {
    static int open_w = 0, open_h = 0, open_d = 0;
    if (open_w != p.width || open_h != p.height || open_d != p.num_disp) {
        check(sva_rows_open(ctx(), &p, rank, world), "sva_rows_open");
        if (world > 1) check(sva_rows_connect_comm(ctx()), "sva_rows_connect_comm");
        open_w = p.width; open_h = p.height; open_d = p.num_disp;
    }
    int32_t by0 = 0, brows = 0;
    check(sva_rows_block(ctx(), &by0, &brows), "sva_rows_block");
    std::vector<sva_image_u8> o;
    for (auto& m : others) o.push_back(view(m));
    sva_image_u8 r = view(ref), mk = mask ? view(*mask) : sva_image_u8{};
    std::vector<uint16_t> disp((size_t)p.width * brows);
    std::vector<float> sub((size_t)p.width * brows);
    check(sva_depth_rows_sharded(ctx(), &p, &r, o.data(), mask ? &mk : nullptr, disp.data(), sub.data()), "svaDepthRowsSharded");
    if (y0) *y0 = by0;
    if (rows) *rows = brows;
    if (subpix) *subpix = sub;
    return disp;
}

// ---- a stream of frames through the row-block pipeline in the order skewed by chain position (sva_rows_stream_*): one call per frame ----
namespace {
void check_ctx(sva_ctx* c, int rc, const char* what) {
    if (rc < 0) throw cv::Exception(std::string(what) + ": " + sva_last_error(c));
}
}  // namespace

SvaRowsStream::SvaRowsStream(int device, const sva_params& p, int rank, int world, const std::array<uint8_t, SVA_COMM_ID_BYTES>* comm_id) {
    try {
        for (int j = 0; j <= world; j++) {
            sva_ctx* c = nullptr;
            const int rc = sva_create(device, &c);
            if (rc != SVA_OK) throw cv::Exception(std::string("sva_create failed (status ") + std::to_string(rc) + "): " + sva_last_error(nullptr));
            ctxs_.push_back(c);
            if (j) {  // one stream for all of them: frames interleave by enqueue order, never as concurrent kernels
                void* s = nullptr;
                check_ctx(ctxs_[0], sva_get_stream(ctxs_[0], &s), "sva_get_stream");
                check_ctx(c, sva_set_stream(c, s), "sva_set_stream");
            }
            check_ctx(c, sva_rows_open(c, &p, rank, world), "sva_rows_open");
        }
        if (world > 1) {
            if (!comm_id) throw cv::Exception("SvaRowsStream: several ranks need the communicator id of svaCommUniqueId");
            check_ctx(ctxs_[0], sva_comm_init(ctxs_[0], comm_id->data(), rank, world), "sva_comm_init");
        }
        check_ctx(ctxs_[0], sva_rows_stream_create(ctxs_.data(), (int32_t)ctxs_.size(), &p, &stream_), "sva_rows_stream_create");
        check_ctx(ctxs_[0], sva_rows_stream_connect_comm(stream_), "sva_rows_stream_connect_comm");
        int32_t y0 = 0, rows = 0;
        check_ctx(ctxs_[0], sva_rows_block(ctxs_[0], &y0, &rows), "sva_rows_block");
        y0_ = y0; rows_ = rows;
    } catch (...) {
        release();
        throw;
    }
}

SvaRowsStream::~SvaRowsStream() {
    if (stream_) sva_rows_stream_flush(stream_);  // the neighbours' frames wait for this rank's parts of them
    release();
}

void SvaRowsStream::release() {
    if (stream_) sva_rows_stream_destroy(stream_);
    stream_ = nullptr;
    for (auto it = ctxs_.rbegin(); it != ctxs_.rend(); ++it) sva_destroy(*it);  // the borrowers first: ctxs_[0] owns the stream
    ctxs_.clear();
}

int64_t SvaRowsStream::submit(const cv::Mat& ref, const std::vector<cv::Mat>& others, const cv::Mat* mask, uint16_t* disp_rows, float* subpix_rows) {
    std::vector<sva_image_u8> o;
    for (auto& m : others) o.push_back(view(m));
    sva_image_u8 r = view(ref), mk = mask ? view(*mask) : sva_image_u8{};
    int64_t ticket = -1;
    check_ctx(ctxs_[0], sva_rows_stream_submit(stream_, &r, o.data(), mask ? &mk : nullptr, disp_rows, subpix_rows, &ticket), "sva_rows_stream_submit");
    return ticket;
}

void SvaRowsStream::flush() { check_ctx(ctxs_[0], sva_rows_stream_flush(stream_), "sva_rows_stream_flush"); }

void SvaRowsStream::wait(int64_t ticket) { check_ctx(ctxs_[0], sva_rows_stream_wait(stream_, ticket), "sva_rows_stream_wait"); }
