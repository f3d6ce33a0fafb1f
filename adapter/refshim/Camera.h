// TEST INFRASTRUCTURE ONLY (adapter/).  Stand-in for the reference's include/Camera.h: the declarations that
// adapter/sva_functions.cpp defines, with the data members in the reference's order (pos3D, f, pixel_size; see sva_camera in
// include/sva_c_api.h).  build_adapter_test.py compiles against it when no reference tree is given, so the adapter's tests run
// from this repository alone.
#pragma once
#include <opencv2/core.hpp>

class Camera {
public:
    Camera(double focal_length, cv::Point3d position, double pixel_size);
    ~Camera();
    cv::Point2i project(cv::Point3d Pos3D);
    cv::Point3d inv_project(cv::Point2i pixel);

    cv::Point3d pos3D;
    double f;
    double pixel_size;
};
