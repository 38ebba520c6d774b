// RetinaFace.cpp -- see RetinaFace.h.  Everything that computes lives behind the C ABI.
#include "RetinaFace.h"

#include <algorithm>
#include <cmath>
#include <cstring>

#include <stdexcept>

RetinaFace::RetinaFace(string &model, string network_, float nms, const RetinaFaceOptions &opt)
    : opt_(opt), network(network_), nms_threshold(nms) {
    // RetinaFace.cpp:211-271: the network-name switch lives behind the C ABI (rf_network_config / rf_config.network); names the
    // reference itself has no anchor configuration for (fmc != 3) or whose models do not ship (net3a) are refused there
    int levels = 0, nratios = 0;
    if (rf_network_config(network.c_str(), &levels, nullptr, nullptr, nullptr, &nratios) != RF_OK)
        throw std::runtime_error("network setting error " + network + ": " + rf_last_error(nullptr));
    const string path = model + "/" + opt_.model_file;
    rf_config cfg{};
    const string table = model + "/" + opt_.int8_table_file;
    const string proto = opt_.prototxt_file.empty() ? string() : model + "/" + opt_.prototxt_file;
    cfg.network = network.c_str();
    cfg.prototxt_path = proto.empty() ? nullptr : proto.c_str();     // buildTrtContext(prototxt, caffemodel), RetinaFace.cpp:276
    cfg.cache_path = opt_.cache_file.empty() ? nullptr : opt_.cache_file.c_str();
    cfg.caffemodel_path = path.c_str();
    cfg.int8_table_path = opt_.precision == RF_PREC_INT8 ? table.c_str() : nullptr;
    cfg.precision = opt_.precision;
    cfg.net_w = opt_.net_w;
    cfg.net_h = opt_.net_h;
    cfg.max_batch = opt_.max_batch;
    cfg.max_faces = opt_.max_faces;
    cfg.device = opt_.device;
    cfg.max_image_w = opt_.max_image_w;
    cfg.max_image_h = opt_.max_image_h;
    int rc = rf_create(&cfg, &h_);
    if (rc != RF_OK) throw std::runtime_error(string("rf_create: ") + rf_status_string(rc) + ": " + rf_last_error(nullptr));
    rf_get_net_size(h_, &opt_.net_w, &opt_.net_h, nullptr, &opt_.max_faces);     // (0 x 0: the prototxt's input size)
    out_faces_.resize((size_t)opt_.max_batch * opt_.max_faces);
    out_counts_.resize(opt_.max_batch);
}

RetinaFace::~RetinaFace() { rf_destroy(h_); }

void RetinaFace::detect(const Mat &img, float threshold, float /*scales*/) {
    if (img.empty()) {   // RetinaFace.cpp:578-580
        last_.clear();
        return;
    }
    vector<cv::Mat> one(1, img);
    detectBatchImages(one, threshold);
}

void RetinaFace::detectEncoded(const vector<vector<unsigned char>> &jpegs, float threshold) {
    last_.assign(jpegs.size(), vector<FaceDetectInfo>());
    scales_.assign(jpegs.size(), 1.f);
    const size_t mb = (size_t)opt_.max_batch;
    for (size_t start = 0; start < jpegs.size(); start += mb) {
        const int n = (int)std::min(mb, jpegs.size() - start);
        vector<const uint8_t *> ptrs(n);
        vector<size_t> lens(n);
        vector<int> ws(n), hs(n);
        for (int i = 0; i < n; i++) { ptrs[i] = jpegs[start + i].data(); lens[i] = jpegs[start + i].size(); }
        int rc = rf_detect_jpeg_batch(h_, ptrs.data(), lens.data(), n, threshold, nms_threshold, out_faces_.data(), out_counts_.data(), nullptr,
                                      ws.data(), hs.data());
        if (rc != RF_OK) throw std::runtime_error(string("rf_detect_jpeg_batch: ") + rf_status_string(rc) + ": " + rf_last_error(h_));
        for (int i = 0; i < n; i++) {
            float sw = 1.0f * ws[i] / opt_.net_w, sh = 1.0f * hs[i] / opt_.net_h;   // RetinaFace.cpp:587-591
            float sc = sw > sh ? sw : sh;
            scales_[start + i] = sc > 1.0f ? sc : 1.0f;
            const FaceDetectInfo *f = reinterpret_cast<const FaceDetectInfo *>(out_faces_.data() + (size_t)i * opt_.max_faces);
            last_[start + i].assign(f, f + out_counts_[i]);
        }
    }
}

void RetinaFace::detectBatchImages(vector<cv::Mat> imgs, float threshold) {
    last_.assign(imgs.size(), vector<FaceDetectInfo>());
    scales_.assign(imgs.size(), 1.f);
    const size_t mb = (size_t)opt_.max_batch;
    for (size_t start = 0; start < imgs.size(); start += mb) {   // the reference asserts n <= maxBatchSize; chunk instead
        const int n = (int)std::min(mb, imgs.size() - start);
        vector<const uint8_t *> ptrs(n);
        vector<int> ws(n), hs(n), strides(n);
        for (int i = 0; i < n; i++) {
            const cv::Mat &m = imgs[start + i];
            if (m.empty()) throw std::runtime_error("detectBatchImages: empty image");
            ptrs[i] = m.data; ws[i] = m.cols; hs[i] = m.rows; strides[i] = (int)m.step;
            float sw = 1.0f * m.cols / opt_.net_w, sh = 1.0f * m.rows / opt_.net_h;   // RetinaFace.cpp:587-591
            float sc = sw > sh ? sw : sh;
            scales_[start + i] = sc > 1.0f ? sc : 1.0f;
        }
        int rc = rf_detect_batch(h_, ptrs.data(), ws.data(), hs.data(), strides.data(), n, threshold, nms_threshold,
                                 out_faces_.data(), out_counts_.data(), nullptr);
        if (rc != RF_OK) throw std::runtime_error(string("rf_detect_batch: ") + rf_status_string(rc) + ": " + rf_last_error(h_));
        for (int i = 0; i < n; i++) {
            const FaceDetectInfo *f = reinterpret_cast<const FaceDetectInfo *>(out_faces_.data() + (size_t)i * opt_.max_faces);
            last_[start + i].assign(f, f + out_counts_[i]);
        }
    }
}

void RetinaFace::detectAndAlign(vector<cv::Mat> imgs, float threshold) {
    last_.assign(imgs.size(), vector<FaceDetectInfo>());
    scales_.assign(imgs.size(), 1.f);
    crops_.assign(imgs.size(), vector<Mat>());
    rf_align_spec spec{};             // zero template: the ArcFace one, scaled by crop_size / 112
    spec.crop_w = spec.crop_h = opt_.crop_size;
    spec.max_crops = opt_.max_crops;
    spec.layout = RF_CROP_U8_BGR;
    const size_t mb = (size_t)opt_.max_batch, crop_bytes = (size_t)opt_.crop_size * opt_.crop_size * 3;
    vector<unsigned char> crops(mb * (size_t)opt_.max_crops * crop_bytes);
    for (size_t start = 0; start < imgs.size(); start += mb) {
        const int n = (int)std::min(mb, imgs.size() - start);
        vector<const uint8_t *> ptrs(n);
        vector<int> ws(n), hs(n), strides(n);
        for (int i = 0; i < n; i++) {
            const cv::Mat &m = imgs[start + i];
            if (m.empty()) throw std::runtime_error("detectAndAlign: empty image");
            ptrs[i] = m.data; ws[i] = m.cols; hs[i] = m.rows; strides[i] = (int)m.step;
        }
        int rc = rf_detect_align_batch(h_, ptrs.data(), ws.data(), hs.data(), strides.data(), n, threshold, nms_threshold, &spec,
                                       out_faces_.data(), out_counts_.data(), nullptr, scales_.data() + start, crops.data(), nullptr);
        if (rc != RF_OK) throw std::runtime_error(string("rf_detect_align_batch: ") + rf_status_string(rc) + ": " + rf_last_error(h_));
        for (int i = 0; i < n; i++) {
            const FaceDetectInfo *f = reinterpret_cast<const FaceDetectInfo *>(out_faces_.data() + (size_t)i * opt_.max_faces);
            last_[start + i].assign(f, f + out_counts_[i]);
            for (int j = 0; j < std::min(out_counts_[i], opt_.max_crops); j++) {
                Mat c(opt_.crop_size, opt_.crop_size, CV_8UC3);
                std::memcpy(c.data, crops.data() + ((size_t)i * opt_.max_crops + j) * crop_bytes, crop_bytes);
                crops_[start + i].push_back(c);
            }
        }
    }
}

vector<FaceDetectInfo> RetinaFace::detectInImage(const Mat &img, float threshold, const vector<float> &scales, bool flip) {
    vector<FaceDetectInfo> out;
    if (img.empty()) return out;
    vector<rf_view> views;
    for (float s : scales) {
        views.push_back(rf_view{s, 0});
        if (flip) views.push_back(rf_view{s, 1});
    }
    int count = 0;
    int rc = rf_detect_views(h_, img.data, img.cols, img.rows, (int)img.step, views.data(), (int)views.size(), threshold, nms_threshold,
                             out_faces_.data(), &count, nullptr, nullptr);
    if (rc != RF_OK) throw std::runtime_error(string("rf_detect_views: ") + rf_status_string(rc) + ": " + rf_last_error(h_));
    const FaceDetectInfo *f = reinterpret_cast<const FaceDetectInfo *>(out_faces_.data());
    out.assign(f, f + count);
    return out;
}

Mat RetinaFace::draw(const Mat &img, const vector<FaceDetectInfo> &faces) {
    Mat out = img.clone();     // RetinaFace.cpp:744: drawing on the caller's image would accumulate boxes
    auto fill = [&out](int x0, int y0, int x1, int y1, unsigned char b, unsigned char g, unsigned char r) {
        x0 = std::max(x0, 0); y0 = std::max(y0, 0); x1 = std::min(x1, out.cols); y1 = std::min(y1, out.rows);
        for (int y = y0; y < y1; y++)
            for (int x = x0; x < x1; x++) {
                unsigned char *p = out.data + (size_t)y * out.step + (size_t)x * 3;
                p[0] = b; p[1] = g; p[2] = r;
            }
    };
    for (const FaceDetectInfo &f : faces) {
        const int x1 = (int)lroundf(f.rect.x1), y1 = (int)lroundf(f.rect.y1), x2 = (int)lroundf(f.rect.x2), y2 = (int)lroundf(f.rect.y2);
        fill(x1 - 1, y1 - 1, x2 + 1, y1 + 1, 0, 0, 255);      // Scalar(0, 0, 255), thickness 2 (:735)
        fill(x1 - 1, y2 - 1, x2 + 1, y2 + 1, 0, 0, 255);
        fill(x1 - 1, y1 - 1, x1 + 1, y2 + 1, 0, 0, 255);
        fill(x2 - 1, y1 - 1, x2 + 1, y2 + 1, 0, 0, 255);
        for (int k = 0; k < 5; k++) {                          // Scalar(0, 255, 0) dots (:739)
            const int cx = (int)lroundf(f.pts.x[k]), cy = (int)lroundf(f.pts.y[k]);
            fill(cx - 1, cy - 1, cx + 2, cy + 2, 0, 255, 0);
        }
    }
    return out;
}
