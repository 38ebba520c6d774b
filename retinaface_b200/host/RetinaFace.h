// RetinaFace.h -- C++ host side of the B200 path: the reference's detector class surface
// (retinaface/RetinaFace.h:15-70) over the C ABI of librf_b200.so (include/rf_b200.h).
//
// Source-compatible with the reference's callers (retinaface/main.cpp:15,43-44):
//     RetinaFace *rf = new RetinaFace(path, "net3");
//     rf->detect(img, 0.9);
//     rf->detectBatchImages(imgs, 0.9);
// Same constructor arguments (model directory, network name, nms threshold), same record types.
// Differences, all additive: the reference's detect functions return void and DROP their result
// (RetinaFace.cpp:665,726,747); here the result is kept and readable through lastFaces() /
// lastBatchFaces(); the network input size, which the reference bakes into prototxt line 7, is a
// constructor option; errors throw std::runtime_error instead of abort()/exit().
#ifndef RF_B200_HOST_RETINAFACE_H
#define RF_B200_HOST_RETINAFACE_H

#include <string>
#include <vector>

#include "cv_compat.hpp"
#include "rf_b200.h"

using namespace std;   // the reference header does this (RetinaFace.h:12); callers rely on it
using cv::Mat;

struct anchor_box { float x1, y1, x2, y2; };               // RetinaFace.h:23-29
struct FacePts { float x[5]; float y[5]; };                // RetinaFace.h:31-35
struct FaceDetectInfo { float score; anchor_box rect; FacePts pts; };   // RetinaFace.h:37-42
static_assert(sizeof(FaceDetectInfo) == sizeof(rf_face), "FaceDetectInfo must match rf_face");

struct RetinaFaceOptions {
    int net_w = 320, net_h = 320;        // the shipped mnet-deconv-0517.prototxt:7 says 320x320
    int max_batch = 8;                   // trtretinafacenet.cpp:21
    int max_faces = 256;
    int precision = RF_PREC_FP16;
    int device = 0;
    int max_image_w = 4096, max_image_h = 3072;   // RetinaFace.cpp:325
    string model_file = "mnet-deconv-0517.caffemodel";   // RetinaFace.cpp:276
    string int8_table_file = "mnet-deconv-0517.table.int8";   // used when precision == RF_PREC_INT8 (trtnetbase.cpp:13)
    string prototxt_file;                // e.g. "mnet-deconv-0517.prototxt" (RetinaFace.cpp:276): parsed, checked, drives the weight
                                         // folding; with net_w = net_h = 0 it also sets the network size.  Empty: built-in graph
    string cache_file;                   // folded-model cache (the reference's "retina.cache", trtnetbase.cpp:205-243, but with a
                                         // staleness check).  Empty: none
    int crop_size = 112;                 // detectAndAlign: side of the aligned crops (a multiple of 112: the ArcFace template)
    int max_crops = 16;                  // detectAndAlign: crops of at most this many top-scoring faces per image
};

class RetinaFace {
   public:
    RetinaFace(string &model, string network = "net3", float nms = 0.4, const RetinaFaceOptions &opt = RetinaFaceOptions());
    ~RetinaFace();
    RetinaFace(const RetinaFace &) = delete;
    RetinaFace &operator=(const RetinaFace &) = delete;

    void detectBatchImages(vector<cv::Mat> imgs, float threshold = 0.5);
    void detect(const Mat &img, float threshold = 0.5, float scales = 1.0);
    // compressed input: what main.cpp:18-26 hands to cv::imread.  The JPEG bitstreams are decoded on the GPU
    // (rf_detect_jpeg_batch); results and lastScale() as for detectBatchImages
    void detectEncoded(const vector<vector<unsigned char>> &jpegs, float threshold = 0.5);

    // detection + the step a recognition pipeline takes next (insightface's norm_crop): for each image, crop_size x crop_size
    // u8 BGR crops of its top max_crops faces, aligned on the GPU by the similarity from their five landmarks to the ArcFace
    // template and sampled from the ORIGINAL image (rf_detect_align_batch; byte-identical to cv::warpAffine with that matrix).
    // Faces and lastScale() as for detectBatchImages; crops of image i in lastCrops(i), in score order.
    void detectAndAlign(vector<cv::Mat> imgs, float threshold = 0.5);
    const vector<Mat> &lastCrops(size_t i = 0) const { return i < crops_.size() ? crops_[i] : no_crops_; }

    // results of the last call, in network-input pixels (RetinaFace.cpp:707); multiply by
    // lastScale() to map back to the caller's image (RetinaFace.cpp:587-591, 732-738)
    const vector<FaceDetectInfo> &lastFaces() const { return last_.empty() ? empty_ : last_[0]; }
    const vector<vector<FaceDetectInfo>> &lastBatchFaces() const { return last_; }
    float lastScale(size_t i = 0) const { return i < scales_.size() ? scales_[i] : 1.f; }
    // SURVEY.md 8f-2 -- what the reference leaves commented out (RetinaFace.cpp:730-746) or unused (`scales`, RetinaFace.h:70):
    // faces of ONE image in ORIGINAL IMAGE pixels (x * scale), optionally with multi-scale / horizontal-flip test-time
    // augmentation: `scales` are fractions (0, 1] of the network input the image is fitted into; with `flip` each scale also
    // runs mirrored.  All views run as one batch and are merged by NMS on the GPU (rf_detect_views).
    vector<FaceDetectInfo> detectInImage(const Mat &img, float threshold = 0.5, const vector<float> &scales = vector<float>(1, 1.0f),
                                         bool flip = false);
    // the reference's visualisation (RetinaFace.cpp:730-741): red box outline (thickness 2), green landmark dots, on a clone
    static Mat draw(const Mat &img, const vector<FaceDetectInfo> &faces);
    int netWidth() const { return opt_.net_w; }
    int netHeight() const { return opt_.net_h; }

   private:
    rf_handle h_ = nullptr;
    RetinaFaceOptions opt_;
    string network;
    float nms_threshold;
    vector<vector<FaceDetectInfo>> last_;
    vector<FaceDetectInfo> empty_;
    vector<float> scales_;
    vector<vector<Mat>> crops_;
    vector<Mat> no_crops_;
    vector<rf_face> out_faces_;
    vector<int> out_counts_;
};

#endif
