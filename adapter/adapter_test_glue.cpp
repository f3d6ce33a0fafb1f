// TEST ONLY: C-callable driver that exercises adapter/sva_functions.cpp the way the reference's main() would — through the
// reference's own function names — on harness images (compiled against oracle/cvshim; see tests/test_gpu_adapter.py).
#include <cstring>
#include <string>

#include "Camera.h"
#include "functions.h"
#include "dlibFaceSelect.h"

#include "sva_c_api.h"
#include "sva_rows_stream.h"

cv::Mat svaMatchLiteral(std::vector<cv::Mat>&, std::vector<Camera>&, std::vector<std::array<int, 2>>&, cv::Mat&, int, double, double);
void svaSelectDevice(int device);
std::array<uint8_t, SVA_COMM_ID_BYTES> svaCommUniqueId();
void svaCommInit(const std::array<uint8_t, SVA_COMM_ID_BYTES>& id, int rank, int world);
std::vector<uint16_t> svaDepthPairSharded(const sva_params&, cv::Mat&, std::vector<cv::Mat>&, cv::Mat*, int, std::vector<float>*);
std::vector<uint16_t> svaDepthRowsSharded(const sva_params&, cv::Mat&, std::vector<cv::Mat>&, cv::Mat*, int, int, int*, int*, std::vector<float>*);
std::vector<std::vector<uint16_t>> svaDepthGroups(const sva_params&, std::vector<cv::Mat>&, const std::vector<std::vector<std::array<int, 2>>>&, int,
                                                  const std::vector<cv::Mat>*, std::vector<std::vector<float>>*);
std::vector<uint16_t> svaFuseMaps(int, int, int, int, const std::vector<int>&, const std::vector<std::vector<uint16_t>>&, const std::vector<std::vector<float>>*,
                                  int, const sva_fuse_params&, const cv::Mat*, std::vector<float>*, std::vector<uint8_t>*);
std::vector<uint16_t> svaDepthGroupsFused(const sva_params&, std::vector<cv::Mat>&, const std::vector<std::vector<std::array<int, 2>>>&, int, int,
                                          const sva_fuse_params&, std::vector<float>*, std::vector<uint8_t>*, const std::vector<cv::Mat>*, const cv::Mat*);

static cv::Mat g_mask;
cv::Mat getFaceMask(cv::Mat&) { return g_mask.clone(); }
cv::Mat getFaceCircle(cv::Mat& m) { return getFaceMask(m); }
static std::string g_err;

extern "C" const char* adapter_last_error() { return g_err.c_str(); }

// mirrors src/CameraStereoVision.cpp:23-47,98-100,112-114 with the loop nest (:49-95) replaced by ONE call
extern "C" int adapter_driver(const uint8_t* const* images25, int w, int h, const uint8_t* mask, uint8_t* out_disp, uint8_t* out_improved, double* out_absdiff) {
    try {
        std::vector<cv::Mat> images;
        for (int i = 0; i < 25; i++) {
            cv::Mat m(h, w, CV_8UC1);
            std::memcpy(m.data, images25[i], (size_t)w * h);
            images.push_back(m);
        }
        g_mask = cv::Mat(h, w, CV_8UC1);
        std::memcpy(g_mask.data, mask, (size_t)w * h);
        double f = 0.05, sensor_size = 0.036, pixelSize = sensor_size / w;
        std::vector<Camera> cameras;
        for (int y = 0; y < 5; y++)
            for (int x = 0; x < 5; x++) cameras.push_back(Camera(f, cv::Point3d{-0.1 + x * 0.05, -0.1 + y * 0.05, -0.75}, pixelSize));
        std::vector<std::array<int, 2>> pairs = getCameraPairs(cameras, MID_LEFT);
        cv::Mat m = getFaceMask(images[12]);
        cv::Mat disparity = svaMatchLiteral(images, cameras, pairs, m, 20, 0.5, 1.0);
        std::memcpy(out_disp, disparity.data, (size_t)w * h);
        std::vector<cv::Mat> inpImages = {images[pairs[0][1]]};
        std::vector<std::array<Camera, 2>> inpCameras = {{cameras[pairs[0][0]], cameras[pairs[0][1]]}};
        cv::Mat improved = improveWithDisparity(disparity, images[pairs[0][0]], inpImages, inpCameras, 21);
        std::memcpy(out_improved, improved.data, (size_t)w * h);
        cv::Mat a = images[12](cv::Rect{cv::Point2i{10, 10}, cv::Point2i{50, 50}}), b = images[11](cv::Rect{cv::Point2i{12, 11}, cv::Point2i{52, 51}});
        *out_absdiff = getAbsDiff(a, b);
        return 0;
    } catch (const std::exception& e) { g_err = e.what(); return -1; }
}

// the consumers of the depth output under their reference names (functions.h:24,28,30,32): warp a depth map, lift it to a cloud, re-project it
extern "C" long long adapter_depth_consumers(const double* depth, int w, int h, int cam_in, int cam_out, double* out_shifted, double* out_cloud,
                                             double* out_map, int* out_group_sizes) {
    try {
        double f = 0.05, sensor_size = 0.036, pixelSize = sensor_size / w;
        std::vector<Camera> cameras;
        for (int y = 0; y < 5; y++)
            for (int x = 0; x < 5; x++) cameras.push_back(Camera(f, cv::Point3d{-0.1 + x * 0.05, -0.1 + y * 0.05, -0.75}, pixelSize));
        cv::Mat d(h, w, CV_64FC1);
        std::memcpy(d.data, depth, sizeof(double) * (size_t)w * h);
        cv::Mat shifted = shiftPerspective2(cameras[cam_in], cameras[cam_out], d);
        std::memcpy(out_shifted, shifted.data, sizeof(double) * (size_t)w * h);
        std::vector<cv::Point3d> cloud = DepthMapToPoints3D(d, cameras[cam_in], cv::Size{w, h});
        for (size_t i = 0; i < cloud.size(); i++) { out_cloud[3 * i] = cloud[i].x; out_cloud[3 * i + 1] = cloud[i].y; out_cloud[3 * i + 2] = cloud[i].z; }
        cv::Mat map = Points3DToDepthMap(cloud, cameras[cam_out], cv::Size{w, h});
        std::memcpy(out_map, map.data, sizeof(double) * (size_t)w * h);
        auto groups = getGroups(cameras, "CHESS");
        for (size_t g = 0; g < groups.size() && g < 16; g++) out_group_sizes[g] = (int)groups[g].size();
        return (long long)cloud.size();
    } catch (const std::exception& e) { g_err = e.what(); return -1; }
}

// a C++ host reaching the multi-GPU entry points through the adapter (world_size ranks, one process each; id = 128 bytes from rank 0's
// adapter_comm_id, distributed by the launcher): pair-sharded frame (map on rank 0) and row-sharded frame (this rank's rows)
extern "C" int adapter_comm_id(uint8_t* out128) {
    try { auto id = svaCommUniqueId(); std::memcpy(out128, id.data(), id.size()); return 0; } catch (const std::exception& e) { g_err = e.what(); return -1; }
}
extern "C" int adapter_multi_gpu(int device, const uint8_t* id128, int rank, int world, const sva_params* p, const uint8_t* ref, const uint8_t* const* others,
                                 uint16_t* out_pairs_disp, uint16_t* out_rows_disp, float* out_rows_sub, int* out_y0, int* out_rows) {
    try {
        svaSelectDevice(device);
        std::array<uint8_t, SVA_COMM_ID_BYTES> id;
        std::memcpy(id.data(), id128, id.size());
        static bool inited = false;
        if (!inited) { svaCommInit(id, rank, world); inited = true; }
        const int w = p->width, h = p->height;
        cv::Mat r(h, w, CV_8UC1);
        std::memcpy(r.data, ref, (size_t)w * h);
        std::vector<cv::Mat> o;
        for (int i = 0; i < p->n_pairs; i++) { cv::Mat m(h, w, CV_8UC1); std::memcpy(m.data, others[i], (size_t)w * h); o.push_back(m); }
        std::vector<uint16_t> d = svaDepthPairSharded(*p, r, o, nullptr, 0, nullptr);
        if (rank == 0) std::memcpy(out_pairs_disp, d.data(), d.size() * 2);
        std::vector<float> sub;
        std::vector<uint16_t> dr = svaDepthRowsSharded(*p, r, o, nullptr, rank, world, out_y0, out_rows, &sub);
        std::memcpy(out_rows_disp, dr.data(), dr.size() * 2);
        std::memcpy(out_rows_sub, sub.data(), sub.size() * 4);
        return 0;
    } catch (const std::exception& e) { g_err = e.what(); return -1; }
}

// a C++ host streaming frames through the row-block pipeline (SvaRowsStream) as rank `rank` of `world`: n frames, frame f = refs[f], the
// n_pairs views others[f * n_pairs ...] and masks[f] (null: no mask); this rank's rows of frame f land at out_disp / out_sub + f * rows * width.
// All frames are submitted, then flushed and waited for in reverse order.
extern "C" int adapter_rows_stream(int device, const uint8_t* id128, int rank, int world, const sva_params* p, int n, const uint8_t* const* refs,
                                   const uint8_t* const* others, const uint8_t* const* masks, uint16_t* out_disp, float* out_sub, int* out_y0, int* out_rows) {
    try {
        const int w = p->width, h = p->height;
        auto mat = [&](const uint8_t* src) { cv::Mat m(h, w, CV_8UC1); std::memcpy(m.data, src, (size_t)w * h); return m; };
        std::array<uint8_t, SVA_COMM_ID_BYTES> id{};
        if (id128) std::memcpy(id.data(), id128, id.size());
        SvaRowsStream s(device, *p, rank, world, id128 ? &id : nullptr);
        std::vector<cv::Mat> ref, msk;
        std::vector<std::vector<cv::Mat>> oth(n);
        for (int f = 0; f < n; f++) {
            ref.push_back(mat(refs[f]));
            msk.push_back(masks[f] ? mat(masks[f]) : cv::Mat());
            for (int i = 0; i < p->n_pairs; i++) oth[f].push_back(mat(others[(size_t)f * p->n_pairs + i]));
        }
        const size_t px = (size_t)s.rows() * w;
        std::vector<int64_t> tickets;
        for (int f = 0; f < n; f++) tickets.push_back(s.submit(ref[f], oth[f], masks[f] ? &msk[f] : nullptr, out_disp + f * px, out_sub + f * px));
        s.flush();
        for (int f = n - 1; f >= 0; f--) s.wait(tickets[f]);
        *out_y0 = s.y0();
        *out_rows = s.rows();
        return 0;
    } catch (const std::exception& e) { g_err = e.what(); return -1; }
}

// the 13 CHESS groups of a 5 x 5 frame the way a reference host gets them: getGroups(cameras, "CHESS") straight into svaDepthGroups.  masks13:
// null, or one pointer per group (null: no mask).  Group g's maps land at out_disp / out_sub + g * w * h.  Returns the number of groups.
extern "C" int adapter_depth_groups(const sva_params* p, const uint8_t* const* images25, const uint8_t* const* masks13, uint16_t* out_disp, float* out_sub) {
    try {
        const int w = p->width, h = p->height;
        auto mat = [&](const uint8_t* src) { cv::Mat m(h, w, CV_8UC1); std::memcpy(m.data, src, (size_t)w * h); return m; };
        double f = 0.05, sensor_size = 0.036, pixelSize = sensor_size / w;
        std::vector<Camera> cameras;
        std::vector<cv::Mat> images;
        for (int y = 0; y < 5; y++)
            for (int x = 0; x < 5; x++) {
                cameras.push_back(Camera(f, cv::Point3d{-0.1 + x * 0.05, -0.1 + y * 0.05, -0.75}, pixelSize));
                images.push_back(mat(images25[5 * y + x]));
            }
        auto groups = getGroups(cameras, "CHESS");
        std::vector<cv::Mat> masks;
        if (masks13)
            for (size_t g = 0; g < groups.size(); g++) masks.push_back(masks13[g] ? mat(masks13[g]) : cv::Mat());
        std::vector<std::vector<float>> sub;
        std::vector<std::vector<uint16_t>> disp = svaDepthGroups(*p, images, groups, 5, masks13 ? &masks : nullptr, &sub);
        const size_t px = (size_t)w * h;
        for (size_t g = 0; g < groups.size(); g++) {
            std::memcpy(out_disp + g * px, disp[g].data(), px * 2);
            std::memcpy(out_sub + g * px, sub[g].data(), px * 4);
        }
        return (int)groups.size();
    } catch (const std::exception& e) { g_err = e.what(); return -1; }
}

// the CHESS groups of a 5 x 5 frame fused into camera target's view, twice: svaDepthGroupsFused(p, images, getGroups(cameras, "CHESS"), 5,
// target, f, &subpix, &support) into out_*[0 .. w * h), and svaDepthGroups followed by svaFuseMaps (sub-pixel maps iff p->subpixel) into
// out_*[w * h .. 2 w * h).  target_mask: null or w x h.  Returns the number of groups.
extern "C" int adapter_depth_groups_fused(const sva_params* p, const uint8_t* const* images25, int target, int tol_16, int min_support,
                                          const uint8_t* target_mask, uint16_t* out_disp, float* out_sub, uint8_t* out_support) {
    try {
        const int w = p->width, h = p->height;
        const size_t px = (size_t)w * h;
        auto mat = [&](const uint8_t* src) { cv::Mat m(h, w, CV_8UC1); std::memcpy(m.data, src, px); return m; };
        double f = 0.05, sensor_size = 0.036, pixelSize = sensor_size / w;
        std::vector<Camera> cameras;
        std::vector<cv::Mat> images;
        for (int y = 0; y < 5; y++)
            for (int x = 0; x < 5; x++) {
                cameras.push_back(Camera(f, cv::Point3d{-0.1 + x * 0.05, -0.1 + y * 0.05, -0.75}, pixelSize));
                images.push_back(mat(images25[5 * y + x]));
            }
        auto groups = getGroups(cameras, "CHESS");
        sva_fuse_params fp{};
        fp.tol_16 = tol_16;
        fp.min_support = min_support;
        cv::Mat tm = target_mask ? mat(target_mask) : cv::Mat();
        std::vector<float> sub;
        std::vector<uint8_t> sup;
        std::vector<uint16_t> d = svaDepthGroupsFused(*p, images, groups, 5, target, fp, &sub, &sup, nullptr, &tm);
        std::memcpy(out_disp, d.data(), px * 2);
        std::memcpy(out_sub, sub.data(), px * 4);
        std::memcpy(out_support, sup.data(), px);
        std::vector<std::vector<float>> gsub;
        std::vector<std::vector<uint16_t>> gdisp = svaDepthGroups(*p, images, groups, 5, nullptr, &gsub);
        std::vector<int> refs;
        for (auto& g : groups) refs.push_back(g[0][0]);
        d = svaFuseMaps(w, h, 5, 25, refs, gdisp, p->subpixel == 1 ? &gsub : nullptr, target, fp, &tm, &sub, &sup);
        std::memcpy(out_disp + px, d.data(), px * 2);
        std::memcpy(out_sub + px, sub.data(), px * 4);
        std::memcpy(out_support + px, sup.data(), px);
        return (int)groups.size();
    } catch (const std::exception& e) { g_err = e.what(); return -1; }
}
