// adapter/sva_rows_stream.h — a C++ host's route to the fastest multi-GPU mode: a stream of frames through the row-block pipeline in the
// order skewed by chain position (sva_rows_stream_*, DESIGN.md §7), one call per frame on cv::Mat images.  Implemented in sva_functions.cpp.
#pragma once
#include <array>
#include <cstdint>
#include <vector>

#include <opencv2/core.hpp>

#include "sva_c_api.h"

class SvaRowsStream {
  public:
    // world + 1 contexts of this rank on `device`, all on one stream, each with a link for this rank's block of rows; the links are connected
    // over ONE communicator (sva_rows_stream_connect_comm).  world > 1: comm_id = svaCommUniqueId() of rank 0, handed to every rank by the
    // launcher; every rank constructs its stream (collective).  Throws cv::Exception on failure.
    SvaRowsStream(int device, const sva_params& p, int rank, int world, const std::array<uint8_t, SVA_COMM_ID_BYTES>* comm_id = nullptr);
    ~SvaRowsStream();  // flushes, then destroys the stream and its contexts
    SvaRowsStream(const SvaRowsStream&) = delete;
    SvaRowsStream& operator=(const SvaRowsStream&) = delete;

    int y0() const { return y0_; }      // this rank's image rows [y0, y0 + rows)
    int rows() const { return rows_; }
    // one frame -> ticket.  disp_rows (rows() x width u16) and subpix_rows (rows() x width f32, may be null) receive this rank's rows in
    // wait(ticket), or when the ticket's slot is reused world + 2 frames later; until then the images and outputs must stay untouched.
    int64_t submit(const cv::Mat& ref, const std::vector<cv::Mat>& others, const cv::Mat* mask, uint16_t* disp_rows, float* subpix_rows);
    void flush();  // every submitted frame completes (every rank makes the same sequence of submit and flush calls)
    void wait(int64_t ticket);

  private:
    std::vector<sva_ctx*> ctxs_;
    sva_rows_stream* stream_ = nullptr;
    int y0_ = 0, rows_ = 0;
    void release();
};
