// TEST INFRASTRUCTURE ONLY (adapter/).  Stand-in for the reference's include/dlibFaceSelect.h: the face-mask ROI that
// improveWithDisparity takes its mask from.  adapter/adapter_test_glue.cpp defines both to return the mask the test registered.
#pragma once
#include <opencv2/core.hpp>

cv::Mat getFaceMask(cv::Mat& sampleImage);
cv::Mat getFaceCircle(cv::Mat& image);
