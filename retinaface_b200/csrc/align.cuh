// align.cuh -- landmark-aligned face crops (the step after detection in a recognition pipeline).
//
// insightface's norm_crop: a similarity transform fitted from a face's five landmarks to a fixed template (estimate_norm,
// Umeyama without reflection), then cv2.warpAffine(img, M, (crop_w, crop_h), INTER_LINEAR, BORDER_CONSTANT, 0).  One launch
// aligns every kept face of a batch: grid (max_crops, n), one CTA per crop slot; the face counts are read from device memory, so
// the launch follows the forward with no host round trip.  Per crop:
//   - landmarks in image pixels: lx * scale in FP32 (the reference's map-back factor, RetinaFace.cpp:587-591, 732-738);
//   - the closed-form least-squares fit of [a -b; b a] + t in FP64 on one thread; the forward matrix (image -> crop, what
//     insightface passes to warpAffine) is written out as 6 doubles;
//   - the warp restates OpenCV's fixed-point arithmetic so that crops are BYTE-IDENTICAL to cv2.warpAffine with that matrix:
//     inversion in OpenCV's operation order, AB_BITS = 10 source coordinates, 5-bit fractions, the initInterTab2D weight table,
//     (sum + (1 << 14)) >> 15, taps outside the image read 0 (compiled with -fmad=false: no contraction changes a rounding).
// Output layouts: RF_CROP_U8_BGR [crop_h][crop_w][3] u8 (norm_crop's output) or RF_CROP_F16_RGB [3][crop_h][crop_w] FP16 of
// (v - mean) * scale, a recognizer's input tensor.
#pragma once
#include "common.cuh"

namespace rf {

constexpr int ALIGN_MAX_CROP = 1024;   // largest crop side

// One source image of the batch: u8 BGR HWC rows of `row_bytes` bytes; `scale` maps network-input pixels to its pixels.
struct AlignSrc {
    const uint8_t *ptr;
    int w, h, row_bytes;
    float scale;
};

struct AlignArgs {
    const AlignSrc *table;        // device [n] or nullptr: image i is `uniform` with ptr + i * uniform_stride
    AlignSrc uniform;
    size_t uniform_stride;
    const rf_det *dets;           // [n][max_faces] records, score order
    const int32_t *counts;        // [n]
    int max_faces, max_crops;
    int crop_w, crop_h, layout;
    float dst_x[5], dst_y[5];     // template in crop pixels
    float mean, scale;            // RF_CROP_F16_RGB
    void *crops;                  // [n][max_crops][crop]
    double *affine;               // [n][max_crops][6] or nullptr
};

// Enqueues the align kernel for images 0..n-1 on `s`.
cudaError_t launch_align(const AlignArgs &a, int n, cudaStream_t s);

}  // namespace rf
