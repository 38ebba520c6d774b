// main.cpp -- the reference's driver (retinaface/main.cpp:14-53) against the B200 class shell:
// construct the detector from a model directory, then time detect() in a loop.  The reference
// loops forever on a hard-coded JPEG; this one takes a raw BGR image (or synthesises noise) and
// a finite iteration count so that it can run unattended.
//   rf_main <model_dir> [--image raw.bgr W H | --jpeg file.jpg] [--net W H] [--iters N] [--batch B] [--thr T] [--tta] [--draw out.bgr]
//           [--align crops.bgr]
// --jpeg is the reference's own input form (main.cpp:18: cv::imread of a JPEG): the file's bytes go to the GPU decoder.
// --align writes the 112 x 112 aligned crops of image 0 (detectAndAlign), one after another, as raw u8 BGR.
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <iostream>
#include <iterator>
#include <vector>

#include "RetinaFace.h"

int main(int argc, char **argv) {
    if (argc < 2) {
        std::fprintf(stderr, "usage: %s <model_dir> [--image raw.bgr W H] [--net W H] [--iters N] [--batch B] [--thr T]\n", argv[0]);
        return 2;
    }
    string path = argv[1];
    RetinaFaceOptions opt;
    opt.net_w = 448; opt.net_h = 448;
    int iters = 1000, batch = 1, iw = 448, ih = 448;
    float thr = 0.9f;
    string image, draw_path, jpeg, align_path;
    bool tta = false;
    for (int i = 2; i < argc; i++) {
        if (!strcmp(argv[i], "--image") && i + 3 < argc) { image = argv[i + 1]; iw = atoi(argv[i + 2]); ih = atoi(argv[i + 3]); i += 3; }
        else if (!strcmp(argv[i], "--jpeg") && i + 1 < argc) jpeg = argv[++i];
        else if (!strcmp(argv[i], "--net") && i + 2 < argc) { opt.net_w = atoi(argv[i + 1]); opt.net_h = atoi(argv[i + 2]); i += 2; }
        else if (!strcmp(argv[i], "--iters") && i + 1 < argc) iters = atoi(argv[++i]);
        else if (!strcmp(argv[i], "--batch") && i + 1 < argc) batch = atoi(argv[++i]);
        else if (!strcmp(argv[i], "--thr") && i + 1 < argc) thr = (float)atof(argv[++i]);
        else if (!strcmp(argv[i], "--model") && i + 1 < argc) opt.model_file = argv[++i];
        else if (!strcmp(argv[i], "--tta")) tta = true;
        else if (!strcmp(argv[i], "--draw") && i + 1 < argc) draw_path = argv[++i];
        else if (!strcmp(argv[i], "--align") && i + 1 < argc) align_path = argv[++i];
    }
    opt.max_batch = batch > opt.max_batch ? batch : opt.max_batch;
    try {
        if (!jpeg.empty()) { opt.max_image_w = 4096; opt.max_image_h = 3072; }
        RetinaFace *rf = new RetinaFace(path, "net3", 0.4, opt);
        if (!jpeg.empty()) {
            std::ifstream f(jpeg, std::ios::binary);
            vector<unsigned char> bytes((std::istreambuf_iterator<char>(f)), std::istreambuf_iterator<char>());
            if (bytes.empty()) { std::fprintf(stderr, "cannot read %s\n", jpeg.c_str()); return 2; }
            vector<vector<unsigned char>> streams(batch, bytes);
            float time = 0;
            for (int it = 0; it < iters; it++) {
                auto t0 = std::chrono::steady_clock::now();
                rf->detectEncoded(streams, thr);
                time += std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t0).count();
            }
            printf("face detection average time = %f ms over %d calls (batch %d, JPEG decoded on the GPU); %zu faces in image 0\n", time / iters, iters, batch,
                   rf->lastFaces().size());
            for (const FaceDetectInfo &f : rf->lastFaces())
                printf("  score %.4f box [%.2f %.2f %.2f %.2f] scale %.3f\n", f.score, f.rect.x1, f.rect.y1, f.rect.x2, f.rect.y2, rf->lastScale());
            delete rf;
            return 0;
        }
        cv::Mat img(ih, iw, CV_8UC3);
        if (!image.empty()) {
            std::ifstream f(image, std::ios::binary);
            if (!f.read((char *)img.data, (std::streamsize)iw * ih * 3)) { std::fprintf(stderr, "cannot read %s\n", image.c_str()); return 2; }
        } else {
            unsigned s = 12345;
            for (size_t i = 0; i < (size_t)iw * ih * 3; i++) { s = s * 1664525u + 1013904223u; img.data[i] = (unsigned char)(s >> 24); }
        }
        vector<cv::Mat> imgs(batch, img);
        float time = 0;
        int count = 0;
        for (int it = 0; it < iters; it++) {
            auto t0 = std::chrono::steady_clock::now();
            if (batch == 1) rf->detect(img, thr); else rf->detectBatchImages(imgs, thr);
            time += std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t0).count();
            count++;
            if (count % 1000 == 0) printf("face detection average time = %f.\n", time / count);
        }
        printf("face detection average time = %f ms over %d calls (batch %d); %zu faces in image 0\n", time / count, count, batch,
               rf->lastFaces().size());
        for (const FaceDetectInfo &f : rf->lastFaces())
            printf("  score %.4f box [%.2f %.2f %.2f %.2f] scale %.3f\n", f.score, f.rect.x1, f.rect.y1, f.rect.x2, f.rect.y2, rf->lastScale());
        if (tta || !draw_path.empty()) {
            // what the reference leaves commented out (RetinaFace.cpp:730-746): faces in image pixels, drawn on a clone;
            // --tta adds a 0.75 scale and mirrored views, merged on the GPU
            vector<float> scales(1, 1.0f);
            if (tta) scales.push_back(0.75f);
            vector<FaceDetectInfo> faces = rf->detectInImage(img, thr, scales, tta);
            printf("in image coordinates (%zu view%s): %zu faces\n", scales.size() * (tta ? 2 : 1), tta ? "s" : "", faces.size());
            for (const FaceDetectInfo &f : faces) printf("  score %.4f box [%.2f %.2f %.2f %.2f]\n", f.score, f.rect.x1, f.rect.y1, f.rect.x2, f.rect.y2);
            if (!draw_path.empty()) {
                cv::Mat vis = RetinaFace::draw(img, faces);
                std::ofstream o(draw_path, std::ios::binary);
                for (int y = 0; y < vis.rows; y++) o.write((const char *)vis.data + (size_t)y * vis.step, (std::streamsize)vis.cols * 3);
            }
        }
        if (!align_path.empty()) {
            rf->detectAndAlign(imgs, thr);
            printf("aligned crops of image 0: %zu (%dx%d u8 BGR) -> %s\n", rf->lastCrops().size(), opt.crop_size, opt.crop_size, align_path.c_str());
            std::ofstream o(align_path, std::ios::binary);
            for (const cv::Mat &c : rf->lastCrops())
                for (int y = 0; y < c.rows; y++) o.write((const char *)c.data + (size_t)y * c.step, (std::streamsize)c.cols * 3);
        }
        delete rf;
    } catch (const std::exception &e) {
        std::fprintf(stderr, "error: %s\n", e.what());
        return 1;
    }
    return 0;
}
