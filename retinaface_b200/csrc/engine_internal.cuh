// engine_internal.cuh -- what the translation units behind include/rf_b200.h share: the handle, the step / tensor records,
// the plan builder, and the functions each unit exports to the others.
//   plan_fp.cu   FP32 / FP16 layer plan (build_plan<T>), tensor-core launch helpers, tile geometry
//   plan_i8.cu   INT8 layer plan (build_plan_i8)
//   engine.cu    tensor placement, CUDA-graph executor, the C-ABI entry points
#pragma once
#include <algorithm>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <functional>
#include <map>
#include <memory>
#include <string>
#include <type_traits>
#include <vector>

#include "align.cuh"
#include "common.cuh"
#include "host_copy.h"
#include "model.h"
#include "postproc.cuh"
#include "preprocess.cuh"

using namespace rf;

#define RF_STR2(x) #x
#define RF_STR(x) RF_STR2(x)

namespace rf_eng {

struct TileChain;                 // plan_tile.cu
std::string &create_error();      // thread-local text of the last failed rf_create (engine.cu)

struct CudaFail { cudaError_t e; const char *what; const char *file; int line; };
// a plan-time failure that is not a CUDA error: carries the rf_status and the full message to rf_create / the caller
struct PlanFail { int status; std::string msg; };
#define CK(call)                                                        \
    do {                                                                \
        cudaError_t _e = (call);                                        \
        if (_e != cudaSuccess) throw CudaFail{_e, #call, __FILE__, __LINE__}; \
    } while (0)

inline std::string fmt(const char *f, ...) {
    char buf[1024];
    va_list ap;
    va_start(ap, f);
    vsnprintf(buf, sizeof buf, f, ap);
    va_end(ap);
    return buf;
}

struct TensorInfo {
    std::string name;
    int h = 0, w = 0, c = 0;
    size_t bytes_per_img = 0;
    int first = -1, last = -1;
    size_t offset = 0;  // bytes into the arena (already scaled by max_batch)
};

struct Step {
    std::string name;
    std::vector<int> in, out;
    std::function<void(int /*n*/, cudaStream_t)> launch;
    double flops_per_img = 0, bytes_per_img = 0;  // algorithmic
    int lane = 0;                 // 0 = main stream; 1, 2 = side branches of the forward graph
    std::vector<int> deps;        // producer steps in OTHER lanes this step must wait for (filled by link_steps)
    bool signals = false;         // some step in another lane waits for this one
};

}  // namespace rf_eng
using namespace rf_eng;

namespace rf_eng {
// multi-GPU exchange state of a handle (comm.cu)
struct Comm {
    int rank = 0, world = 1, ring = 0;
    bool ready = false;
    unsigned char *window = nullptr;       // this rank's gather window (device)
    size_t bytes = 0;
    unsigned char *peer[RF_COMM_MAX_WORLD] = {nullptr};
    bool opened[RF_COMM_MAX_WORLD] = {false};
    unsigned seq = 0;                      // steps exchanged so far
    unsigned *d_err = nullptr, *h_err = nullptr;
    unsigned char blob[128] = {0};
    struct Slot { rf_det *h_dets = nullptr; int *h_counts = nullptr; } slots[RF_PIPELINE_DEPTH];   // pinned, [world][max_batch]...
};
}  // namespace rf_eng

struct rf_handle_s {
    rf_config cfg{};
    rf_eng::Comm comm;
    std::string caffemodel, table;
    std::string err;
    Model model;
    std::map<std::string, float> int8_scales;
    int device = 0;
    int elem = 4;  // bytes per activation element
    cudaStream_t stream = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;

    std::vector<TensorInfo> tensors;
    std::map<std::string, int> tensor_by_name;
    std::vector<Step> steps;
    int head_step = -1, nms_step = -1;
    std::vector<std::shared_ptr<TileChain>> chains;   // tile-chain launches of the FP16 plan (plan_tile.cu)
    unsigned tile_mask = 0;                           // which parts of the FP16 plan run as tile chains (RF_TILE_MASK)
    int lane_last[3] = {-1, -1, -1};                  // last step of each side lane (joined at the end of the forward)
    int cache_status = 0;                             // model.h CACHE_*: how the folded model was obtained
    bool profiling = false;                           // rf_profile_layers is launching single steps out of their forward
    int tile_expected = 0;                            // tiles per image over the three SSH chains (last-block NMS)
    std::vector<float> tile_bias_tmp;                 // plan-time scratch
    unsigned *tile_dbg = nullptr, *tile_dbg_dev = nullptr;   // host-mapped word a timed-out hand-off of a tile chain reports into
    unsigned char *arena = nullptr;
    size_t arena_bytes = 0;

    // weights
    std::vector<float> wstage;  // host staging of all fp32 weights
    float *d_weights = nullptr;
    std::vector<__half> wstage_h;  // FP16 tensor-core weight images (tc_conv.cuh B chunks)
    __half *d_weights_h = nullptr;
    std::vector<int8_t> wstage_q;  // INT8 tensor-core weight images (tc_conv_i8.cuh)
    int8_t *d_weights_q = nullptr;
    bool use_tc = false;

    // io
    uint8_t *d_input = nullptr;       // [max_batch][H][W][3] u8 BGR
    uint8_t *h_input = nullptr;       // pinned mirror
    PostBuffers pb_merge{};           // rf_detect_views: candidates of all views of one image (lazily allocated)
    uint8_t *d_raw = nullptr;         // one raw caller image (max_image) for the letterbox kernel
    uint8_t *h_raw = nullptr;         // pinned, TWO buffers of raw_bytes: staging of pageable caller images (upload_raw)
    size_t raw_bytes = 0;
    int raw_slots = 1;                // raw device buffers (one per batch element, capped)
    cudaEvent_t raw_ev[2] = {nullptr, nullptr};   // H2D out of staging buffer i has completed
    unsigned raw_seq = 0;
    std::unique_ptr<HostCopyPool> copy_pool;      // row-band parallel host copy into the staging buffers (lazily created)
    PostParams *d_params = nullptr, *h_params = nullptr;
    PostBuffers pb{};
    LevelDesc lv[3];
    HeadWeights hw[3];
    int feat_tensor[3] = {-1, -1, -1};
    float *d_blobs[9] = {nullptr};    // rf_forward_heads / rf_postprocess staging (device)
    size_t blob_elems[9] = {0};       // per image
    rf_det *h_dets = nullptr;         // pinned [max_batch][max_faces]
    int *h_counts = nullptr;          // pinned [2*max_batch]: kept, candidates
    std::map<int, cudaGraphExec_t> graphs;
    // aligned crops of rf_detect_align_batch (context 0; lazily allocated, regrown when a spec needs more)
    uint8_t *d_crops = nullptr;       // [max_batch][max_crops][crop]
    double *d_affine = nullptr;       // [max_batch][max_crops][6]
    size_t crops_bytes = 0, affine_count = 0;
    AlignSrc *d_align_src = nullptr, *h_align_src = nullptr;   // [max_batch] source table of the align kernel (device, pinned)
    // pipelined end-to-end path (rf_submit_batch / rf_collect_batch)
    struct Slot {
        uint8_t *d_in = nullptr, *h_in = nullptr;     // device input, pinned staging for pageable sources
        rf_det *h_dets = nullptr;                      // pinned results
        int *h_counts = nullptr;
        cudaEvent_t ev_h2d = nullptr, ev_done = nullptr;
        int n = 0;
        bool busy = false, gather = false;
    } slots[RF_PIPELINE_DEPTH];
    cudaStream_t copy_stream = nullptr;
    unsigned submit_seq = 0, collect_seq = 0;
    cudaStream_t lane_stream[3] = {nullptr, nullptr, nullptr};   // [0] unused (the caller's stream is lane 0)
    std::vector<cudaEvent_t> step_event;
    bool blobs_in_plan = false;       // head step writes blobs (forward_heads path)
    static constexpr int kParamSlots = 1024;
    unsigned param_seq = 0;
    float cur_thr = 0.5f, cur_nms = 0.4f;

    void *tptr(int id) const { return arena + tensors[id].offset; }

    // Execution contexts.  Everything a forward pass writes (activation arena, candidate / output buffers,
    // run parameters) and everything it is issued on (stream, lane streams, events, captured graphs) exists
    // once per context; the asynchronous entry points rotate through the contexts so that consecutive batches
    // overlap on the GPU (most kernels of one batch-8 step fill well under one wave of the 148 SMs).  The
    // members above always hold the ACTIVE context; switch_ctx() swaps them with a saved one.
    struct Ctx {
        cudaStream_t stream = nullptr, lane_stream[3] = {nullptr, nullptr, nullptr};
        std::vector<cudaEvent_t> step_event;
        unsigned char *arena = nullptr;
        PostBuffers pb{};
        PostParams *d_params = nullptr, *h_params = nullptr;
        unsigned param_seq = 0;
        float cur_thr = 0.5f, cur_nms = 0.4f;
        std::map<int, cudaGraphExec_t> graphs;
        cudaEvent_t fence = nullptr;
    };
    std::vector<Ctx> saved;
    int active = 0, nctx = 1;
    unsigned next_dev_ctx = 0;
    cudaStream_t last_stream = nullptr;
    cudaEvent_t fence = nullptr;
    void *jpeg = nullptr;             // nvJPEG decoder state (jpeg.cu), created by the first JPEG call
};

namespace rf_eng {
inline void switch_ctx(rf_handle h, int i) {
    if (i == h->active) return;
    auto xchg = [&](rf_handle_s::Ctx &c) {
        std::swap(c.stream, h->stream);
        for (int l = 0; l < 3; l++) std::swap(c.lane_stream[l], h->lane_stream[l]);
        std::swap(c.step_event, h->step_event);
        std::swap(c.arena, h->arena);
        std::swap(c.pb, h->pb);
        std::swap(c.d_params, h->d_params);
        std::swap(c.h_params, h->h_params);
        std::swap(c.param_seq, h->param_seq);
        std::swap(c.cur_thr, h->cur_thr);
        std::swap(c.cur_nms, h->cur_nms);
        std::swap(c.graphs, h->graphs);
        std::swap(c.fence, h->fence);
    };
    xchg(h->saved[h->active]);   // park the active state in its slot
    xchg(h->saved[i]);           // and bring context i in
    h->active = i;
}

inline int fail(rf_handle h, int code, const std::string &msg) {
    if (h) h->err = msg; else create_error() = msg;
    return code;
}
inline int fail_cuda(rf_handle h, const CudaFail &f) {
    std::string extra;
    if (h && h->tile_dbg && h->tile_dbg[0])
        extra = fmt(" [tile chain: CTA %u timed out waiting at tile_chain.cuh:%u]", h->tile_dbg[0] >> 20, h->tile_dbg[0] & 0xfffffu);
    return fail(h, RF_ERR_CUDA, fmt("%s failed: %s (%s:%d)%s", f.what, cudaGetErrorString(f.e), f.file, f.line, extra.c_str()));
}

// ---------------------------------------------------------------------------------------------
// Plan builder
// ---------------------------------------------------------------------------------------------
struct Builder {
    rf_handle h;
    int H, W;
    size_t add_weights(const std::vector<float> &v) {
        size_t off = h->wstage.size();
        h->wstage.insert(h->wstage.end(), v.begin(), v.end());
        while (h->wstage.size() % 4) h->wstage.push_back(0.f);  // keep float4 alignment
        return off;
    }
    size_t add_weights_h(const std::vector<__half> &v) {
        size_t off = h->wstage_h.size();
        h->wstage_h.insert(h->wstage_h.end(), v.begin(), v.end());
        while (h->wstage_h.size() % 64) h->wstage_h.push_back(__float2half(0.f));  // 128-byte alignment for bulk copies
        return off;
    }
    size_t add_weights_q(const std::vector<int8_t> &v) {
        size_t off = h->wstage_q.size();
        h->wstage_q.insert(h->wstage_q.end(), v.begin(), v.end());
        while (h->wstage_q.size() % 128) h->wstage_q.push_back(0);
        return off;
    }
    int tensor(const std::string &name, int hh, int ww, int c) {
        TensorInfo t;
        t.name = name; t.h = hh; t.w = ww; t.c = c;
        t.bytes_per_img = (size_t)hh * ww * c * h->elem;
        h->tensors.push_back(t);
        h->tensor_by_name[name] = (int)h->tensors.size() - 1;
        return (int)h->tensors.size() - 1;
    }
    void step(Step s) { h->steps.push_back(std::move(s)); }
};

// ---- exported by plan_fp.cu -----------------------------------------------------------------------------------------
constexpr int TC_SMEM_LIMIT = 200 * 1024;   // dynamic shared memory the tensor-core kernels may opt into (they also hold ~5 KB static)
struct DwGeom { int rows, nsplit, Rmax; };
template <typename T>
void build_plan(rf_handle h);               // T = float (RF_PREC_FP32) | __half (RF_PREC_FP16)
cudaError_t tc_init();
std::vector<__half> make_stem_blob(const std::vector<float> &w0, const std::vector<float> &b0, const std::vector<float> &wd,
                                   const std::vector<float> &bd, const std::vector<float> &wp, const std::vector<float> &bp);
int plan_stem_tc(Builder &B);
int plan_pair_legacy(Builder &B, int i, int tin, int ih, int iw);
void plan_conv_legacy(Builder &B, const std::string &sname, std::vector<const FoldedConv *> cs, int tin, int ih, int iw, int t0, int ld0,
                      int off0, int n0, int relu0, int t1, int ld1, int off1, int relu1, int lane = 0, int tup = -1, int up_which = 0);
int plan_fpn_merge_h2(Builder &B, const std::string &name, int tlat, int tup, int fh, int fw, int which);
template <typename T>
void plan_heads_and_nms(Builder &B, bool with_heads, bool with_nms);
std::vector<__half> pack_tc_weights(const std::vector<const FoldedConv *> &cs, std::vector<float> &bias, int &Kpad, int nsplit = 1);
// ---- exported by plan_tile.cu ---------------------------------------------------------------------------------------
void build_plan_tiles(rf_handle h);         // RF_PREC_FP16 with tensor cores: tile chains (tile_chain.cuh) + round-1 kernels where no chain fits
cudaError_t tile_init();
std::string describe_chains(rf_handle h);
// ---- exported by comm.cu --------------------------------------------------------------------------------------------
void comm_release(rf_handle h);
void comm_wait_in_graph(rf_handle h, int n, cudaStream_t s);   // last node of the forward once a communicator exists
// ---- exported by jpeg.cu (f1 ingest: nvJPEG decode into device memory) ------------------------------------------------
int jpeg_info(rf_handle h, const uint8_t *data, size_t len, int *w, int *hgt);
int jpeg_decode(rf_handle h, const uint8_t *const *data, const size_t *len, int n, uint8_t *const *dst, const int *w, const int *hgt, cudaStream_t s);
void jpeg_release(rf_handle h);
const char *jpeg_backend(rf_handle h);
// ---- exported by plan_i8.cu -----------------------------------------------------------------------------------------
void build_plan_i8(rf_handle h);
cudaError_t tc_init_i8();

}  // namespace rf_eng
