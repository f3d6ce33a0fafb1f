// TEST INFRASTRUCTURE ONLY (adapter/).  Stand-in for the reference's include/functions.h: the signatures that
// adapter/sva_functions.cpp implements, and enum pairType with the values of sva_pair_type (include/sva_c_api.h).
#pragma once
#include <array>
#include <string>
#include <vector>

#include <opencv2/core.hpp>

#include "Camera.h"

enum pairType { ORTHOGONAL, DIAGONAL, TO_CENTER, LINE_HORIZONTAL, LINE_VERTICAL, CROSS, JUMP_CROSS, TO_CENTER_SMALL, MID_LEFT, MID_TOP };

cv::Mat improveWithDisparity(cv::Mat& disparity, cv::Mat centerImage, std::vector<cv::Mat>& images, std::vector<std::array<Camera, 2>>& cameras,
                             int windowSize);
cv::Mat shiftPerspective2(Camera inputCam, Camera outputCam, cv::Mat& depthMap);
cv::Mat shiftPerspectiveWithDisparity(Camera& inputCam, Camera& outputCam, cv::Mat& disparity, cv::Mat& image);
cv::Mat Points3DToDepthMap(std::vector<cv::Point3d>& points, Camera camera, cv::Size resolution);
std::vector<cv::Point3d> DepthMapToPoints3D(cv::Mat& depthMap, Camera camera, cv::Size resolution);
std::vector<std::array<int, 2>> getCameraPairs(const std::vector<Camera>& cameras, const pairType pairs);
std::vector<std::array<int, 2>> getCameraPairs(const std::vector<Camera>& cameras, const pairType pair, int cameraNum);
std::vector<std::vector<std::array<int, 2>>> getGroups(std::vector<Camera>& cameras, std::string groupType);
double getAbsDiff(cv::Mat& mat1, cv::Mat& mat2);
std::vector<cv::Point2i> bresenham(cv::Point2i point1, cv::Point2i point2);
