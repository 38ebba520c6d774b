// engine.cu -- the handle behind include/rf_b200.h: model upload, activation arena, CUDA-graph executor and the C-ABI entry
// points.  The layer plans live in plan_fp.cu (FP32 / FP16) and plan_i8.cu (INT8); shared types in engine_internal.cuh.
//
// Replaces the reference's engine slot: TrtNetBase / TrtRetinaFaceNet
// (retinaface/tensorrt/trtnetbase.cpp:199-330, trtretinafacenet.cpp:48-210) and the detect
// orchestration of RetinaFace::detect / detectBatchImages (retinaface/RetinaFace.cpp:576-940).
#include "engine_internal.cuh"
#include "align.cuh"
#include "calibrate.cuh"
#include "preprocess.cuh"

namespace rf_eng {

std::string &create_error() {
    thread_local std::string text;
    return text;
}

// Cross-lane dependencies: a step waits (event) for the producers of its inputs that live in another lane.
void link_steps(rf_handle h) {
    auto &st = h->steps;
    for (int i = 0; i < (int)st.size(); i++) {
        st[i].deps.clear();
        for (int t : st[i].in) {
            for (int j = i - 1; j >= 0; j--) {
                bool writes = false;
                for (int o : st[j].out) writes |= (o == t);
                if (!writes) continue;
                if (st[j].lane != st[i].lane) {
                    if (std::find(st[i].deps.begin(), st[i].deps.end(), j) == st[i].deps.end()) st[i].deps.push_back(j);
                    st[j].signals = true;
                }
                break;   // the last writer before i (its lane orders earlier writers of the same tensor)
            }
        }
    }
    // the forward ends on the main lane: side lanes whose last step nobody waits for (SSH chains with fused predictors)
    // are joined explicitly at the end of run_steps
    for (int l = 1; l < 3; l++) {
        h->lane_last[l] = -1;
        for (int i = 0; i < (int)st.size(); i++) if (st[i].lane == l) h->lane_last[l] = i;
        if (h->lane_last[l] >= 0) st[h->lane_last[l]].signals = true;
    }
}

// Liveness-based first-fit placement of activation tensors in one arena.  Steps on side lanes run
// concurrently with later main-lane steps: every tensor such a step touches stays live until the
// first step of another lane that waits for its lane (the join), so no concurrent writer can land on it.
void place_tensors(rf_handle h, bool keep_all) {
    auto &ts = h->tensors;
    auto &st = h->steps;
    for (int si = 0; si < (int)st.size(); si++) {
        for (int t : st[si].out) { if (ts[t].first < 0) ts[t].first = si; ts[t].last = std::max(ts[t].last, si); }
        for (int t : st[si].in) ts[t].last = std::max(ts[t].last, si);
    }
    for (int k = 0; k < (int)st.size(); k++) {
        if (st[k].lane == 0) continue;
        int join = (int)st.size() - 1;
        for (int j = k + 1; j < (int)st.size() && join == (int)st.size() - 1; j++)
            for (int d : st[j].deps)
                if (st[j].lane != st[k].lane && st[d].lane == st[k].lane && d >= k) { join = j; break; }
        for (int t : st[k].in) ts[t].last = std::max(ts[t].last, join);
        for (int t : st[k].out) ts[t].last = std::max(ts[t].last, join);
    }
    // a main-lane step that runs while a side lane is still reading must not overwrite those inputs either:
    // covered above because the side step's inputs stay live until the join.
    const size_t B = (size_t)h->cfg.max_batch;
    size_t top = 0;
    std::vector<int> order(ts.size());
    for (size_t i = 0; i < ts.size(); i++) order[i] = (int)i;
    std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return ts[a].first < ts[b].first; });
    std::vector<int> placed;
    for (int id : order) {
        size_t sz = (ts[id].bytes_per_img * B + 255) / 256 * 256;
        size_t off = 0;
        if (keep_all) {
            off = top;
        } else {
            bool moved = true;
            while (moved) {
                moved = false;
                for (int p : placed) {
                    bool live_overlap = !(ts[p].last < ts[id].first || ts[id].last < ts[p].first);
                    size_t psz = (ts[p].bytes_per_img * B + 255) / 256 * 256;
                    bool mem_overlap = off < ts[p].offset + psz && ts[p].offset < off + sz;
                    if (live_overlap && mem_overlap) { off = ts[p].offset + psz; moved = true; }
                }
            }
        }
        ts[id].offset = off;
        top = std::max(top, off + sz);
        placed.push_back(id);
    }
    h->arena_bytes = top;
}

// Issue the forward pass: lane 0 on `s`, side lanes on their own streams, joined by events.  Works both
// under stream capture (the side streams fork from / join into the capturing stream) and eagerly.
void run_steps(rf_handle h, int n, cudaStream_t s, bool use_lanes = true) {
    static const bool one_lane = [] { const char *e = getenv("RF_ONE_LANE"); return e && e[0] == '1'; }();   // A/B measurements
    if (one_lane) use_lanes = false;
    for (size_t i = 0; i < h->steps.size(); i++) {
        Step &st = h->steps[i];
        cudaStream_t cs = (use_lanes && st.lane) ? h->lane_stream[st.lane] : s;
        if (use_lanes)
            for (int d : st.deps) CK(cudaStreamWaitEvent(cs, h->step_event[d], 0));
        st.launch(n, cs);
        if (use_lanes && st.signals) CK(cudaEventRecord(h->step_event[i], cs));
    }
    if (use_lanes)
        for (int l = 1; l < 3; l++)
            if (h->lane_last[l] >= 0) CK(cudaStreamWaitEvent(s, h->step_event[h->lane_last[l]], 0));
    // multi-GPU handles: the wait for every rank's records of this step is the forward's last node (a no-op kernel for runs
    // without an exchange), not a separate launch behind the graph
    if (h->comm.ready && !h->profiling) comm_wait_in_graph(h, n, s);
}

void forward_graph(rf_handle h, int n) {
    if (h->cfg.flags & RF_FLAG_NO_GRAPH) {
        run_steps(h, n, h->stream);
        CK(cudaGetLastError());
        return;
    }
    auto it = h->graphs.find(n);
    if (it == h->graphs.end()) {
        cudaGraph_t g = nullptr;
        CK(cudaStreamBeginCapture(h->stream, cudaStreamCaptureModeThreadLocal));
        run_steps(h, n, h->stream);
        cudaError_t e = cudaStreamEndCapture(h->stream, &g);
        if (e != cudaSuccess) throw CudaFail{e, "cudaStreamEndCapture", __FILE__, __LINE__};
        cudaGraphExec_t ge = nullptr;
        e = cudaGraphInstantiate(&ge, g, 0);
        cudaGraphDestroy(g);
        if (e != cudaSuccess) throw CudaFail{e, "cudaGraphInstantiate", __FILE__, __LINE__};
        it = h->graphs.emplace(n, ge).first;
    }
    CK(cudaGraphLaunch(it->second, h->stream));
}

// Run parameters travel through a small ring of pinned slots so that an asynchronous caller
// (rf_detect_batch_device) can queue several runs without overwriting a copy still in flight.
void set_params(rf_handle h, float thr, float nms, const uint8_t *input = nullptr, unsigned comm_seq = 0) {
    PostParams *slot = h->h_params + (h->param_seq++ % rf_handle_s::kParamSlots);
    slot->score_thr = thr;
    slot->nms_thr = nms;
    slot->input = input ? input : h->d_input;
    slot->comm_seq = comm_seq;
    slot->comm_slot = comm_seq ? comm_seq % (unsigned)h->comm.ring : 0u;
    h->cur_thr = thr;
    h->cur_nms = nms;
    CK(cudaMemcpyAsync(h->d_params, slot, sizeof(PostParams), cudaMemcpyHostToDevice, h->stream));
}

void destroy(rf_handle h) {
    if (!h) return;
    cudaSetDevice(h->device);
    if (h->saved.empty()) h->saved.resize(1);
    for (int c = 0; c < (int)h->saved.size(); c++) { switch_ctx(h, c); if (h->stream) cudaStreamSynchronize(h->stream); }
    comm_release(h);
    jpeg_release(h);
    for (int c = 0; c < (int)h->saved.size(); c++) {
        switch_ctx(h, c);
        if (h->stream) cudaStreamSynchronize(h->stream);
        for (auto &g : h->graphs) cudaGraphExecDestroy(g.second);
        h->graphs.clear();
        cudaFree(h->arena); cudaFree(h->d_params); cudaFreeHost(h->h_params);
        cudaFree(h->pb.cand_keys); cudaFree(h->pb.cand_recs); cudaFree(h->pb.cand_count); cudaFree(h->pb.sort_scratch);
        cudaFree(h->pb.flag_scratch); cudaFree(h->pb.out_dets); cudaFree(h->pb.out_counts); cudaFree(h->pb.out_total_kept); cudaFree(h->pb.tile_done);
        for (auto e : h->step_event) if (e) cudaEventDestroy(e);
        for (int l = 1; l < 3; l++) if (h->lane_stream[l]) cudaStreamDestroy(h->lane_stream[l]);
        if (h->fence) cudaEventDestroy(h->fence);
        if (h->stream) cudaStreamDestroy(h->stream);
    }
    cudaFree(h->pb_merge.cand_keys); cudaFree(h->pb_merge.cand_recs); cudaFree(h->pb_merge.cand_count); cudaFree(h->pb_merge.sort_scratch);
    cudaFree(h->pb_merge.flag_scratch); cudaFree(h->pb_merge.out_dets); cudaFree(h->pb_merge.out_counts); cudaFree(h->pb_merge.out_total_kept);
    cudaFree(h->d_weights); cudaFree(h->d_weights_h); cudaFree(h->d_weights_q); cudaFree(h->d_input); cudaFree(h->d_raw);
    for (auto p : h->d_blobs) cudaFree(p);
    h->copy_pool.reset();
    for (auto e : h->raw_ev) if (e) cudaEventDestroy(e);
    cudaFree(h->d_crops); cudaFree(h->d_affine); cudaFree(h->d_align_src); cudaFreeHost(h->h_align_src);
    cudaFreeHost(h->h_input); cudaFreeHost(h->h_raw); cudaFreeHost(h->h_dets); cudaFreeHost(h->h_counts); cudaFreeHost(h->tile_dbg);
    for (auto &sl : h->slots) {
        cudaFree(sl.d_in); cudaFreeHost(sl.h_in); cudaFreeHost(sl.h_dets); cudaFreeHost(sl.h_counts);
        if (sl.ev_h2d) cudaEventDestroy(sl.ev_h2d);
        if (sl.ev_done) cudaEventDestroy(sl.ev_done);
    }
    if (h->copy_stream) cudaStreamDestroy(h->copy_stream);
    if (h->ev0) cudaEventDestroy(h->ev0);
    if (h->ev1) cudaEventDestroy(h->ev1);
    delete h;
}

int check_n(rf_handle h, int n) {
    if (!h) return RF_ERR_INVALID_ARG;
    if (n < 0) return fail(h, RF_ERR_INVALID_ARG, "negative batch size");
    if (n > h->cfg.max_batch) return fail(h, RF_ERR_CAPACITY, fmt("batch %d exceeds max_batch %d", n, h->cfg.max_batch));
    return RF_OK;
}

}  // namespace rf_eng

// =============================================================================================
// C ABI
// =============================================================================================
extern "C" {

int rf_abi_version(void) { return RF_B200_ABI_VERSION; }

const char *rf_build_info(void) {
    return "librf_b200 (RetinaFace mnet25 detect path) built for sm_100a, CUDA " RF_STR(CUDART_VERSION);
}

const char *rf_status_string(int s) {
    switch (s) {
        case RF_OK: return "ok";
        case RF_ERR_INVALID_ARG: return "invalid argument";
        case RF_ERR_IO: return "i/o error";
        case RF_ERR_MODEL: return "model error";
        case RF_ERR_CUDA: return "CUDA error";
        case RF_ERR_NO_DEVICE: return "no usable CUDA device (the library has no CPU path)";
        case RF_ERR_CAPACITY: return "capacity exceeded";
        case RF_ERR_UNSUPPORTED: return "unsupported";
    }
    return "unknown status";
}

const char *rf_last_error(rf_handle h) { return h ? h->err.c_str() : create_error().c_str(); }

int rf_create(const rf_config *cfg, rf_handle *out) {
    if (out) *out = nullptr;
    if (!cfg || !out) return fail(nullptr, RF_ERR_INVALID_ARG, "rf_create: cfg and out must be non-NULL");
    if (!cfg->caffemodel_path) return fail(nullptr, RF_ERR_INVALID_ARG, "rf_create: caffemodel_path is NULL");
    rf_config cfg_local = *cfg;
    NetGraph graph;
    Model model;
    int cache_status = CACHE_NONE;
    {
        // model front end first: the prototxt may supply the network size (trtnetbase.cpp:163-187 reads it from there too)
        std::string err;
        int st = RF_OK;
        if (cfg->network) {
            NetworkConfig nc;
            if (!network_config(cfg->network, nc, err)) return fail(nullptr, RF_ERR_UNSUPPORTED, "rf_create: " + err);
            if (nc.ratios.size() != 1) return fail(nullptr, RF_ERR_UNSUPPORTED, fmt("rf_create: network '%s' uses %zu anchor ratios per scale; the shipped models (and this engine) have 2 anchors per position", cfg->network, nc.ratios.size()));
        }
        if (!load_model(cfg->caffemodel_path, cfg->prototxt_path ? cfg->prototxt_path : "", cfg->cache_path ? cfg->cache_path : "", model, &graph, &cache_status, err, st))
            return fail(nullptr, st, err);
        if (cfg->prototxt_path && cfg_local.net_w == 0 && cfg_local.net_h == 0) { cfg_local.net_h = graph.input_dims[2]; cfg_local.net_w = graph.input_dims[3]; }
    }
    cfg = &cfg_local;
    if (cfg->net_w <= 0 || cfg->net_h <= 0 || cfg->net_w % 32 || cfg->net_h % 32)
        return fail(nullptr, RF_ERR_INVALID_ARG, fmt("rf_create: net size %dx%d must be positive multiples of 32", cfg->net_w, cfg->net_h));
    if (cfg->max_batch <= 0 || cfg->max_batch > 4096) return fail(nullptr, RF_ERR_INVALID_ARG, "rf_create: max_batch must be in [1, 4096]");
    {
        // The kernels index activations with 32-bit element offsets (and pack (image row) << 12 | column in the FPN merge):
        // the largest tensor of a batch -- the stem output, (H/2) x (W/2) x 16 -- must stay below 2^31 elements.
        const long long stem_elems = (long long)cfg->max_batch * (cfg->net_h / 2) * (cfg->net_w / 2) * 16;
        const long long merge_rows = (long long)cfg->max_batch * (cfg->net_h / 8);
        if (stem_elems > 0x7fffffffLL || merge_rows >= (1LL << 19) || cfg->net_w / 8 >= (1 << 12))
            return fail(nullptr, RF_ERR_CAPACITY, fmt("rf_create: max_batch %d at %dx%d exceeds the 32-bit activation index range (largest tensor: %lld elements); "
                                                      "use a smaller max_batch", cfg->max_batch, cfg->net_w, cfg->net_h, stem_elems));
    }
    if (cfg->precision != RF_PREC_FP32 && cfg->precision != RF_PREC_FP16 && cfg->precision != RF_PREC_INT8)
        return fail(nullptr, RF_ERR_INVALID_ARG, "rf_create: unknown precision");
    if (cfg->precision == RF_PREC_INT8 && !cfg->int8_table_path)
        return fail(nullptr, RF_ERR_INVALID_ARG, "rf_create: RF_PREC_INT8 needs int8_table_path (the TensorRT calibration cache of this caffemodel)");

    std::unique_ptr<rf_handle_s, void (*)(rf_handle)> H(new rf_handle_s, destroy);
    rf_handle h = H.get();
    h->cfg = *cfg;
    h->caffemodel = cfg->caffemodel_path;
    h->cfg.caffemodel_path = h->caffemodel.c_str();
    if (cfg->int8_table_path) { h->table = cfg->int8_table_path; h->cfg.int8_table_path = h->table.c_str(); }
    if (h->cfg.max_faces <= 0) h->cfg.max_faces = 256;
    if (h->cfg.max_faces > 8192) return fail(nullptr, RF_ERR_INVALID_ARG, "rf_create: max_faces must be <= 8192");
    if (h->cfg.max_image_w <= 0) h->cfg.max_image_w = h->cfg.net_w;
    if (h->cfg.max_image_h <= 0) h->cfg.max_image_h = h->cfg.net_h;
    h->cfg.max_image_w = std::max(h->cfg.max_image_w, h->cfg.net_w);
    h->cfg.max_image_h = std::max(h->cfg.max_image_h, h->cfg.net_h);
    h->device = cfg->device;
    h->elem = cfg->precision == RF_PREC_FP32 ? 4 : (cfg->precision == RF_PREC_FP16 ? 2 : 1);

    // ---- model (host) --------------------------------------------------------------------
    {
        std::string err;
        h->model = std::move(model);
        h->cache_status = cache_status;
        h->cfg.prototxt_path = h->cfg.cache_path = h->cfg.network = nullptr;     // (the caller's strings are not kept)
        if (!h->table.empty() && !read_int8_table(h->table, h->int8_scales, err)) return fail(nullptr, RF_ERR_IO, err);
    }
    // ---- device ----------------------------------------------------------------------------
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0)
        return fail(nullptr, RF_ERR_NO_DEVICE, fmt("no CUDA device (%s); librf_b200 has no CPU path", e == cudaSuccess ? "count 0" : cudaGetErrorString(e)));
    if (cfg->device < 0 || cfg->device >= ndev) return fail(nullptr, RF_ERR_INVALID_ARG, fmt("device %d out of range (%d devices)", cfg->device, ndev));
    try {
        CK(cudaSetDevice(h->device));
        cudaDeviceProp prop;
        CK(cudaGetDeviceProperties(&prop, h->device));
        if (prop.major != 10)
            return fail(nullptr, RF_ERR_NO_DEVICE, fmt("device %d is sm_%d%d; librf_b200 is built for sm_100a only", h->device, prop.major, prop.minor));
        CK(cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking));
        CK(cudaEventCreate(&h->ev0));
        CK(cudaEventCreate(&h->ev1));
        CK(postproc_init());

        const int Hn = h->cfg.net_h, Wn = h->cfg.net_w, Bm = h->cfg.max_batch;
        // levels / anchors
        const int strides[3] = {32, 16, 8};
        int abase = 0, pbase = 0;
        for (int l = 0; l < 3; l++) {
            LevelDesc &lv = h->lv[l];
            lv.stride = strides[l]; lv.h = Hn / strides[l]; lv.w = Wn / strides[l];
            lv.anchor_base = abase; lv.pix_base = pbase;
            base_anchors_net3(strides[l], lv.base);
            abase += 2 * lv.h * lv.w; pbase += lv.h * lv.w;
        }
        const int A = abase;
        int ap2 = 1;
        while (ap2 < A) ap2 <<= 1;

        h->use_tc = h->cfg.precision == RF_PREC_INT8 || (h->cfg.precision == RF_PREC_FP16 && !(h->cfg.flags & RF_FLAG_NO_TENSORCORE));
        if (h->use_tc) CK(tc_init());
        if (h->cfg.precision == RF_PREC_INT8) { CK(tc_init_i8()); build_plan_i8(h); }
        else if (h->cfg.precision == RF_PREC_FP32) build_plan<float>(h);
        else if (h->use_tc && !(h->cfg.flags & RF_FLAG_LEGACY_TC)) { CK(tile_init()); build_plan_tiles(h); }
        else build_plan<__half>(h);
        link_steps(h);
        place_tensors(h, false);
        CK(cudaMalloc(&h->d_weights, h->wstage.size() * sizeof(float)));
        CK(cudaMemcpy(h->d_weights, h->wstage.data(), h->wstage.size() * sizeof(float), cudaMemcpyHostToDevice));
        if (!h->wstage_h.empty()) {
            CK(cudaMalloc(&h->d_weights_h, h->wstage_h.size() * sizeof(__half)));
            CK(cudaMemcpy(h->d_weights_h, h->wstage_h.data(), h->wstage_h.size() * sizeof(__half), cudaMemcpyHostToDevice));
        }
        if (!h->wstage_q.empty()) {
            CK(cudaMalloc(&h->d_weights_q, h->wstage_q.size()));
            CK(cudaMemcpy(h->d_weights_q, h->wstage_q.data(), h->wstage_q.size(), cudaMemcpyHostToDevice));
        }
        const size_t in_bytes = (size_t)Bm * Hn * Wn * 3;
        CK(cudaMalloc(&h->d_input, in_bytes));
        CK(cudaHostAlloc(&h->h_input, in_bytes, cudaHostAllocDefault));
        h->raw_bytes = ((size_t)h->cfg.max_image_w * h->cfg.max_image_h * 3 + 255) / 256 * 256;
        // one raw buffer per batch element (capped at 2 GiB in total): the images of a call are uploaded back to back and
        // letter-boxed by ONE launch
        h->raw_slots = (int)std::max<size_t>(1, std::min<size_t>((size_t)Bm, ((size_t)2 << 30) / h->raw_bytes));
        CK(cudaMalloc(&h->d_raw, h->raw_bytes * h->raw_slots));
        CK(cudaHostAlloc(&h->h_raw, 2 * h->raw_bytes, cudaHostAllocDefault));
        for (auto &e : h->raw_ev) CK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        CK(cudaHostAlloc(&h->h_dets, sizeof(rf_det) * (size_t)Bm * h->cfg.max_faces, cudaHostAllocDefault));
        CK(cudaHostAlloc(&h->h_counts, sizeof(int) * 2 * Bm, cudaHostAllocDefault));
        CK(cudaHostAlloc(&h->tile_dbg, 64, cudaHostAllocMapped));
        memset(h->tile_dbg, 0, 64);
        CK(cudaHostGetDevicePointer(&h->tile_dbg_dev, h->tile_dbg, 0));
        // ---- per-context resources ----
        h->nctx = h->cfg.streams <= 0 ? RF_MAX_STREAMS : std::min(h->cfg.streams, RF_MAX_STREAMS);
        h->saved.resize(h->nctx);
        for (int c = 0; c < h->nctx; c++) {
            switch_ctx(h, c);
            if (c > 0) CK(cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking));   // context 0 keeps the stream created above
            for (int l = 1; l < 3; l++) CK(cudaStreamCreateWithFlags(&h->lane_stream[l], cudaStreamNonBlocking));
            h->step_event.assign(h->steps.size(), nullptr);
            for (size_t i = 0; i < h->steps.size(); i++)
                if (h->steps[i].signals) CK(cudaEventCreateWithFlags(&h->step_event[i], cudaEventDisableTiming));
            CK(cudaEventCreateWithFlags(&h->fence, cudaEventDisableTiming));
            CK(cudaMalloc(&h->arena, h->arena_bytes));
            CK(cudaMalloc(&h->d_params, sizeof(PostParams)));
            CK(cudaHostAlloc(&h->h_params, sizeof(PostParams) * rf_handle_s::kParamSlots, cudaHostAllocDefault));
            PostBuffers &pb = h->pb;
            pb.anchors_per_image = A; pb.anchors_pow2 = ap2; pb.max_faces = h->cfg.max_faces; pb.max_batch = Bm;
            CK(cudaMalloc(&pb.cand_keys, sizeof(unsigned long long) * (size_t)Bm * A));
            CK(cudaMalloc(&pb.cand_recs, sizeof(rf_det) * (size_t)Bm * A));
            CK(cudaMalloc(&pb.cand_count, sizeof(int) * Bm));
            CK(cudaMemset(pb.cand_count, 0, sizeof(int) * Bm));
            CK(cudaMalloc(&pb.sort_scratch, sizeof(unsigned long long) * (size_t)Bm * ap2));
            CK(cudaMalloc(&pb.flag_scratch, (size_t)Bm * ap2));
            CK(cudaMalloc(&pb.out_dets, sizeof(rf_det) * (size_t)Bm * pb.max_faces));
            CK(cudaMalloc(&pb.out_counts, sizeof(int) * Bm));
            CK(cudaMalloc(&pb.out_total_kept, sizeof(int) * Bm));
            CK(cudaMemset(pb.out_counts, 0, sizeof(int) * Bm));
            CK(cudaMalloc(&pb.tile_done, sizeof(int) * Bm));
            CK(cudaMemset(pb.tile_done, 0, sizeof(int) * Bm));
        }
        switch_ctx(h, 0);
        for (int l = 0; l < 3; l++) {
            const int ch[3] = {4, 8, 20};
            for (int k = 0; k < 3; k++) h->blob_elems[3 * l + k] = (size_t)ch[k] * h->lv[l].h * h->lv[l].w;
        }
        CK(cudaDeviceSynchronize());
    } catch (const CudaFail &f) {
        return fail_cuda(nullptr, f);
    } catch (const PlanFail &f) {
        return fail(nullptr, f.status, "rf_create: " + f.msg);
    }
    *out = H.release();
    return RF_OK;
}

void rf_destroy(rf_handle h) { destroy(h); }

uint8_t *rf_pinned_input(rf_handle h) { return h ? h->h_input : nullptr; }
uint8_t *rf_device_input(rf_handle h) { return h ? h->d_input : nullptr; }

int rf_get_net_size(rf_handle h, int *net_w, int *net_h, int *max_batch, int *max_faces) {
    if (!h) return RF_ERR_INVALID_ARG;
    if (net_w) *net_w = h->cfg.net_w;
    if (net_h) *net_h = h->cfg.net_h;
    if (max_batch) *max_batch = h->cfg.max_batch;
    if (max_faces) *max_faces = h->cfg.max_faces;
    return RF_OK;
}
int rf_num_anchors(rf_handle h) { return h ? h->pb.anchors_per_image : RF_ERR_INVALID_ARG; }
void *rf_stream(rf_handle h) { if (!h) return nullptr; switch_ctx(h, 0); return (void *)h->stream; }

int rf_synchronize(rf_handle h) {
    if (!h) return RF_ERR_INVALID_ARG;
    try {
        CK(cudaSetDevice(h->device));
        const int keep = h->active;
        for (int c = 0; c < h->nctx; c++) { switch_ctx(h, c); CK(cudaStreamSynchronize(h->stream)); }
        switch_ctx(h, keep);
    } catch (const CudaFail &f) { return fail_cuda(h, f); }
    return RF_OK;
}

// Orders context 0's stream (the one rf_stream returns) after everything queued so far on every context.
int rf_fence(rf_handle h) {
    if (!h) return RF_ERR_INVALID_ARG;
    try {
        CK(cudaSetDevice(h->device));
        switch_ctx(h, 0);
        cudaStream_t s0 = h->stream;
        for (int c = 1; c < h->nctx; c++) {
            switch_ctx(h, c);
            CK(cudaEventRecord(h->fence, h->stream));
            CK(cudaStreamWaitEvent(s0, h->fence, 0));
        }
        switch_ctx(h, 0);
    } catch (const CudaFail &f) { return fail_cuda(h, f); }
    return RF_OK;
}

void *rf_last_stream(rf_handle h) { return h ? (void *)(h->last_stream ? h->last_stream : h->stream) : nullptr; }

int rf_launches_per_batch(rf_handle h, int n) {
    (void)n;
    return h ? (int)h->steps.size() : RF_ERR_INVALID_ARG;
}

static int detect_device_impl(rf_handle h, const uint8_t *dev_bgr, int n, float thr, float nms, const rf_det **dev_dets, const int32_t **dev_counts,
                              bool gather) {
    int rc = check_n(h, n);
    if (rc) return rc;
    if (gather && (!h->comm.ready || n == 0)) return fail(h, RF_ERR_INVALID_ARG, "rf_detect_batch_device_allgather: call rf_comm_init first (and n > 0)");
    try {
        CK(cudaSetDevice(h->device));
        switch_ctx(h, (int)(h->next_dev_ctx++ % (unsigned)h->nctx));   // consecutive batches overlap on different contexts
        h->last_stream = h->stream;
        // the caller's device images are read in place (conv0 takes the pointer from the run parameters)
        if (h->param_seq && h->param_seq % rf_handle_s::kParamSlots == 0) CK(cudaStreamSynchronize(h->stream));
        const unsigned seq = gather ? ++h->comm.seq : 0u;
        set_params(h, thr, nms, dev_bgr, seq);
        if (n > 0) forward_graph(h, n);
        if (gather) {
            const unsigned slot = seq % (unsigned)h->comm.ring;
            const size_t img0 = (size_t)slot * h->comm.world * h->cfg.max_batch;
            if (dev_dets) *dev_dets = h->pb.comm.dets[h->comm.rank] + img0 * h->cfg.max_faces;
            if (dev_counts) *dev_counts = h->pb.comm.counts[h->comm.rank] + img0;
            return RF_OK;
        }
    } catch (const CudaFail &f) { return fail_cuda(h, f); }
    if (dev_dets) *dev_dets = h->pb.out_dets;
    if (dev_counts) *dev_counts = h->pb.out_counts;
    return RF_OK;
}

int rf_detect_batch_device(rf_handle h, const uint8_t *dev_bgr, int n, float thr, float nms, const rf_det **dev_dets,
                           const int32_t **dev_counts) {
    return detect_device_impl(h, dev_bgr, n, thr, nms, dev_dets, dev_counts, false);
}
int rf_detect_batch_device_allgather(rf_handle h, const uint8_t *dev_bgr, int n, float thr, float nms, const rf_det **all_dets,
                                     const int32_t **all_counts) {
    return detect_device_impl(h, dev_bgr, n, thr, nms, all_dets, all_counts, true);
}

static int fetch_results(rf_handle h, int n, rf_face *out_faces, int *out_counts, int32_t *out_idx, int *out_ncand) {
    const int mf = h->cfg.max_faces;
    CK(cudaMemcpyAsync(h->h_counts, h->pb.out_counts, sizeof(int) * n, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaMemcpyAsync(h->h_dets, h->pb.out_dets, sizeof(rf_det) * (size_t)n * mf, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    for (int i = 0; i < n; i++) {
        int k = h->h_counts[i];
        if (out_counts) out_counts[i] = k;
        for (int j = 0; j < k; j++) {
            const rf_det &d = h->h_dets[(size_t)i * mf + j];
            if (out_faces) out_faces[(size_t)i * mf + j] = d.face;
            if (out_idx) out_idx[(size_t)i * mf + j] = d.anchor_index;
        }
    }
    (void)out_ncand;
    return RF_OK;
}

// One caller image of arbitrary size -> d_raw (packed rows) on the handle's stream.  Pinned sources (cudaHostAlloc /
// cudaHostRegister) are copied straight from the caller's memory, row stride and all.  Pageable sources are staged through
// two pinned buffers: a row-band parallel host copy (host_copy.h) into one buffer overlaps the DMA out of the other; the
// only host wait is for the DMA that last read the buffer about to be overwritten.  In both cases the stream orders the
// copy into d_raw behind the letter-box kernel that still reads the previous image.
static uint8_t *upload_raw(rf_handle h, const uint8_t *src, int width, int height, int row_stride, int raw_slot = 0) {
    uint8_t *d_dst = h->d_raw + (size_t)raw_slot * h->raw_bytes;
    cudaPointerAttributes at{};
    const bool pinned = cudaPointerGetAttributes(&at, src) == cudaSuccess && at.type == cudaMemoryTypeHost;
    if (pinned) {
        CK(cudaMemcpy2DAsync(d_dst, (size_t)width * 3, src, (size_t)row_stride, (size_t)width * 3, (size_t)height, cudaMemcpyHostToDevice, h->stream));
        return d_dst;
    }
    cudaGetLastError();
    if (!h->copy_pool) h->copy_pool.reset(new HostCopyPool((int)std::min(3u, std::max(1u, std::thread::hardware_concurrency()) - 1u)));
    const int slot = (int)(h->raw_seq++ & 1u);
    uint8_t *buf = h->h_raw + (size_t)slot * h->raw_bytes;
    CK(cudaEventSynchronize(h->raw_ev[slot]));      // (returns at once for an event never recorded)
    h->copy_pool->copy_rows(buf, src, (size_t)width * 3, (size_t)row_stride, height);
    CK(cudaMemcpyAsync(d_dst, buf, (size_t)width * height * 3, cudaMemcpyHostToDevice, h->stream));
    CK(cudaEventRecord(h->raw_ev[slot], h->stream));
    return d_dst;
}

// Input staging of one call of caller images (rf_detect_batch, rf_detect_align_batch) into d_input on the handle's stream.
// Network-sized packed images are copied H2D straight from the caller's memory when it is pinned (cudaHostAlloc /
// cudaHostRegister / the library's own rf_pinned_input), otherwise via the library's pinned mirror; runs of adjacent sources
// collapse into one copy.  Other sizes are uploaded into per-image raw buffers and letter-boxed by ONE launch for all of them
// (preprocess.cuh; RF_FLAG_NPP_RESIZE: the reference's NPP super-sampling definition instead of its OpenCV bilinear one).
// More than raw_slots letter-boxed images reuse the raw buffers chunk by chunk.  srcs / scales (optional, [n]): where each
// image's original pixels are on the device -- still there after the forward only when no raw buffer was reused, which
// rf_detect_align_batch checks before it calls this -- and the reference's map-back factor.
static int stage_inputs(rf_handle h, const char *who, const uint8_t *const *imgs, const int *widths, const int *heights,
                        const int *row_strides, int n, AlignSrc *srcs, float *scales) {
    const int Hn = h->cfg.net_h, Wn = h->cfg.net_w;
    const size_t img_bytes = (size_t)Hn * Wn * 3;
    const uint8_t *run_src = nullptr;
    int run_start = -1, run_len = 0;
    auto flush = [&]() {
        if (run_start < 0) return;
        CK(cudaMemcpyAsync(h->d_input + (size_t)run_start * img_bytes, run_src, (size_t)run_len * img_bytes,
                           cudaMemcpyHostToDevice, h->stream));
        run_start = -1;
    };
    bool staging_dirty = false;
    const int area = (h->cfg.flags & RF_FLAG_NPP_RESIZE) ? 1 : 0;
    std::vector<LbItem> lb;
    auto flush_lb = [&]() {
        if (lb.empty()) return;
        CK(launch_letterbox_batch(lb.data(), (int)lb.size(), Wn, Hn, h->stream));
        lb.clear();
    };
    for (int i = 0; i < n; i++) {
        if (!imgs[i] || widths[i] <= 0 || heights[i] <= 0) { return fail(h, RF_ERR_INVALID_ARG, fmt("%s: image %d is empty", who, i)); }
        const int rs = row_strides && row_strides[i] ? row_strides[i] : widths[i] * 3;
        if (widths[i] == Wn && heights[i] == Hn && rs == Wn * 3) {
            const uint8_t *src = imgs[i];
            const bool in_mirror = src >= h->h_input && src < h->h_input + (size_t)h->cfg.max_batch * img_bytes;
            if (!in_mirror) {
                cudaPointerAttributes at{};
                bool pinned = cudaPointerGetAttributes(&at, src) == cudaSuccess && at.type == cudaMemoryTypeHost;
                if (!pinned) {
                    cudaGetLastError();
                    if (!staging_dirty) { CK(cudaStreamSynchronize(h->stream)); staging_dirty = true; }
                    uint8_t *slot = h->h_input + (size_t)i * img_bytes;
                    memcpy(slot, src, img_bytes);
                    src = slot;
                }
            }
            if (run_start >= 0 && src == run_src + (size_t)run_len * img_bytes) { run_len++; }
            else { flush(); run_start = i; run_src = src; run_len = 1; }
            if (srcs) srcs[i] = AlignSrc{h->d_input + (size_t)i * img_bytes, Wn, Hn, Wn * 3, 1.f};
            if (scales) scales[i] = 1.f;
        } else {
            flush();
            if (widths[i] > h->cfg.max_image_w || heights[i] > h->cfg.max_image_h)
                return fail(h, RF_ERR_CAPACITY, fmt("image %d is %dx%d, larger than max_image %dx%d", i, widths[i], heights[i],
                                                    h->cfg.max_image_w, h->cfg.max_image_h));
            if ((int)lb.size() == h->raw_slots) flush_lb();
            const uint8_t *d_src = upload_raw(h, imgs[i], widths[i], heights[i], rs, (int)lb.size());
            lb.emplace_back();
            const float sc = letterbox_fill(lb.back(), d_src, widths[i], heights[i], h->d_input + (size_t)i * img_bytes, Wn, Hn, 0, area);
            if (srcs) srcs[i] = AlignSrc{d_src, widths[i], heights[i], widths[i] * 3, sc};
            if (scales) scales[i] = sc;
        }
    }
    flush();
    flush_lb();
    return RF_OK;
}

int rf_detect_batch(rf_handle h, const uint8_t *const *imgs, const int *widths, const int *heights, const int *row_strides,
                    int n, float thr, float nms, rf_face *out_faces, int *out_counts, int32_t *out_idx) {
    int rc = check_n(h, n);
    if (rc) return rc;
    if (n == 0) return RF_OK;
    if (!imgs || !widths || !heights) return fail(h, RF_ERR_INVALID_ARG, "rf_detect_batch: NULL image arrays");
    try {
        CK(cudaSetDevice(h->device));
        switch_ctx(h, 0);
        if ((rc = stage_inputs(h, "rf_detect_batch", imgs, widths, heights, row_strides, n, nullptr, nullptr))) return rc;
        set_params(h, thr, nms);
        forward_graph(h, n);
        fetch_results(h, n, out_faces, out_counts, out_idx, nullptr);
    } catch (const CudaFail &f) { return fail_cuda(h, f); }
    return RF_OK;
}

// ---- aligned face crops (align.cuh) -------------------------------------------------------------------------------------------
// insightface's ArcFace template (arcface_dst, float32) of a 112 x 112 crop
static const float kArcface112[5][2] = {{38.2946f, 51.6963f}, {73.5318f, 51.5014f}, {56.0252f, 71.7366f}, {41.5493f, 92.3655f}, {70.7299f, 92.2041f}};

// Checks a spec and fills the geometry / template / layout part of the kernel arguments.
static int align_args(rf_handle h, const char *who, const rf_align_spec *spec, AlignArgs &a) {
    if (!spec) return fail(h, RF_ERR_INVALID_ARG, fmt("%s: NULL rf_align_spec", who));
    if (spec->crop_w <= 0 || spec->crop_h <= 0 || spec->crop_w > ALIGN_MAX_CROP || spec->crop_h > ALIGN_MAX_CROP)
        return fail(h, RF_ERR_INVALID_ARG, fmt("%s: crop %dx%d, each side must be in 1..%d", who, spec->crop_w, spec->crop_h, ALIGN_MAX_CROP));
    if (spec->max_crops < 1 || spec->max_crops > h->cfg.max_faces)
        return fail(h, RF_ERR_INVALID_ARG, fmt("%s: max_crops %d outside 1..max_faces (%d)", who, spec->max_crops, h->cfg.max_faces));
    if (spec->layout != RF_CROP_U8_BGR && spec->layout != RF_CROP_F16_RGB)
        return fail(h, RF_ERR_INVALID_ARG, fmt("%s: unknown crop layout %d", who, spec->layout));
    a = AlignArgs{};
    bool zero = true;
    for (int k = 0; k < 5; k++) zero = zero && spec->dst_x[k] == 0.f && spec->dst_y[k] == 0.f;
    if (zero) {
        if (spec->crop_w % 112 || spec->crop_h % 112)
            return fail(h, RF_ERR_INVALID_ARG, fmt("%s: the default (ArcFace) template needs crop sides that are multiples of 112, got %dx%d; "
                                                   "pass a template for other sizes", who, spec->crop_w, spec->crop_h));
        const float fx = (float)(spec->crop_w / 112.0), fy = (float)(spec->crop_h / 112.0);   // estimate_norm: template * size / 112
        for (int k = 0; k < 5; k++) { a.dst_x[k] = kArcface112[k][0] * fx; a.dst_y[k] = kArcface112[k][1] * fy; }
    } else {
        for (int k = 0; k < 5; k++) { a.dst_x[k] = spec->dst_x[k]; a.dst_y[k] = spec->dst_y[k]; }
    }
    a.crop_w = spec->crop_w; a.crop_h = spec->crop_h; a.layout = spec->layout;
    a.max_crops = spec->max_crops; a.max_faces = h->cfg.max_faces;
    a.mean = spec->mean; a.scale = spec->scale;
    return RF_OK;
}

static size_t crop_bytes(const AlignArgs &a) { return (size_t)a.crop_w * a.crop_h * 3 * (a.layout == RF_CROP_F16_RGB ? 2 : 1); }

int rf_detect_align_batch(rf_handle h, const uint8_t *const *imgs, const int *widths, const int *heights, const int *row_strides, int n,
                          float thr, float nms, const rf_align_spec *spec, rf_face *out_faces, int *out_counts, int32_t *out_idx,
                          float *out_scales, void *out_crops, double *out_affine) {
    static const char *who = "rf_detect_align_batch";
    int rc = check_n(h, n);
    if (rc) return rc;
    AlignArgs a;
    if ((rc = align_args(h, who, spec, a))) return rc;
    if (n == 0) return RF_OK;
    if (!imgs || !widths || !heights || !out_crops) return fail(h, RF_ERR_INVALID_ARG, fmt("%s: NULL image arrays or out_crops", who));
    // the crops are sampled from the raw buffers after the forward: every letter-boxed image of the call needs its own
    int lettered = 0;
    for (int i = 0; i < n; i++) {
        const int rs = row_strides && row_strides[i] ? row_strides[i] : widths[i] * 3;
        lettered += !(widths[i] == h->cfg.net_w && heights[i] == h->cfg.net_h && rs == h->cfg.net_w * 3);
    }
    if (lettered > h->raw_slots)
        return fail(h, RF_ERR_CAPACITY, fmt("%s: %d images are not network-sized; the handle keeps at most %d original images on the device "
                                            "(raw_slots: max_batch, capped at 2 GiB of max_image buffers)", who, lettered, h->raw_slots));
    const size_t cb = crop_bytes(a);
    try {
        CK(cudaSetDevice(h->device));
        switch_ctx(h, 0);
        const size_t slots = (size_t)h->cfg.max_batch * a.max_crops;
        if (slots * cb > h->crops_bytes || slots > h->affine_count) {
            CK(cudaStreamSynchronize(h->stream));
            CK(cudaFree(h->d_crops)); h->d_crops = nullptr;
            CK(cudaFree(h->d_affine)); h->d_affine = nullptr;
            h->crops_bytes = std::max(h->crops_bytes, slots * cb);
            h->affine_count = std::max(h->affine_count, slots);
            CK(cudaMalloc(&h->d_crops, h->crops_bytes));
            CK(cudaMalloc(&h->d_affine, sizeof(double) * 6 * h->affine_count));
        }
        if (!h->d_align_src) {
            CK(cudaMalloc(&h->d_align_src, sizeof(AlignSrc) * h->cfg.max_batch));
            CK(cudaHostAlloc(&h->h_align_src, sizeof(AlignSrc) * h->cfg.max_batch, cudaHostAllocDefault));
        }
        std::vector<float> scales(n);
        if ((rc = stage_inputs(h, who, imgs, widths, heights, row_strides, n, h->h_align_src, scales.data()))) return rc;
        CK(cudaMemcpyAsync(h->d_align_src, h->h_align_src, sizeof(AlignSrc) * n, cudaMemcpyHostToDevice, h->stream));
        set_params(h, thr, nms);
        forward_graph(h, n);
        a.table = h->d_align_src;
        a.dets = h->pb.out_dets;
        a.counts = h->pb.out_counts;
        a.crops = h->d_crops;
        a.affine = h->d_affine;
        CK(launch_align(a, n, h->stream));
        fetch_results(h, n, out_faces, out_counts, out_idx, nullptr);
        // only the crops that exist cross PCIe
        for (int i = 0; i < n; i++) {
            const size_t k = (size_t)std::min(h->h_counts[i], a.max_crops), c0 = (size_t)i * a.max_crops;
            if (!k) continue;
            CK(cudaMemcpyAsync(static_cast<uint8_t *>(out_crops) + c0 * cb, h->d_crops + c0 * cb, k * cb, cudaMemcpyDeviceToHost, h->stream));
            if (out_affine) CK(cudaMemcpyAsync(out_affine + c0 * 6, h->d_affine + c0 * 6, k * 6 * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
        }
        CK(cudaStreamSynchronize(h->stream));
        if (out_scales) for (int i = 0; i < n; i++) out_scales[i] = scales[i];
    } catch (const CudaFail &f) { return fail_cuda(h, f); }
    return RF_OK;
}

int rf_align_batch_device(rf_handle h, const uint8_t *dev_bgr, int n, const rf_det *dev_dets, const int32_t *dev_counts,
                          const rf_align_spec *spec, void *dev_crops, double *dev_affine) {
    static const char *who = "rf_align_batch_device";
    int rc = check_n(h, n);
    if (rc) return rc;
    AlignArgs a;
    if ((rc = align_args(h, who, spec, a))) return rc;
    if (n == 0) return RF_OK;
    if (!dev_bgr || !dev_dets || !dev_counts || !dev_crops) return fail(h, RF_ERR_INVALID_ARG, fmt("%s: NULL device pointer", who));
    const int Hn = h->cfg.net_h, Wn = h->cfg.net_w;
    try {
        CK(cudaSetDevice(h->device));
        a.table = nullptr;
        a.uniform = AlignSrc{dev_bgr, Wn, Hn, Wn * 3, 1.f};
        a.uniform_stride = (size_t)Hn * Wn * 3;
        a.dets = dev_dets;
        a.counts = dev_counts;
        a.crops = dev_crops;
        a.affine = dev_affine;
        CK(launch_align(a, n, h->last_stream ? h->last_stream : h->stream));   // the stream rf_last_stream() reports
    } catch (const CudaFail &f) { return fail_cuda(h, f); }
    return RF_OK;
}

// ---- f1 ingest: compressed images (main.cpp:18-26 decodes on the host with cv::imread) ---------------------------------------
int rf_detect_jpeg_batch(rf_handle h, const uint8_t *const *jpegs, const size_t *jpeg_bytes, int n, float thr, float nms, rf_face *out_faces,
                         int *out_counts, int32_t *out_idx, int *out_widths, int *out_heights) {
    int rc = check_n(h, n);
    if (rc) return rc;
    if (n == 0) return RF_OK;
    if (!jpegs || !jpeg_bytes) return fail(h, RF_ERR_INVALID_ARG, "rf_detect_jpeg_batch: NULL stream arrays");
    const int Hn = h->cfg.net_h, Wn = h->cfg.net_w;
    const size_t img_bytes = (size_t)Hn * Wn * 3;
    try {
        CK(cudaSetDevice(h->device));
        switch_ctx(h, 0);
        std::vector<int> w(n), hg(n);
        for (int i = 0; i < n; i++) {
            if (!jpegs[i] || !jpeg_bytes[i]) return fail(h, RF_ERR_INVALID_ARG, fmt("rf_detect_jpeg_batch: stream %d is empty", i));
            if ((rc = jpeg_info(h, jpegs[i], jpeg_bytes[i], &w[i], &hg[i]))) return rc;
            if (w[i] <= 0 || hg[i] <= 0 || w[i] > h->cfg.max_image_w || hg[i] > h->cfg.max_image_h)
                return fail(h, RF_ERR_CAPACITY, fmt("JPEG %d is %dx%d, larger than max_image %dx%d", i, w[i], hg[i], h->cfg.max_image_w, h->cfg.max_image_h));
            if (out_widths) out_widths[i] = w[i];
            if (out_heights) out_heights[i] = hg[i];
        }
        const int area = (h->cfg.flags & RF_FLAG_NPP_RESIZE) ? 1 : 0;
        // network-sized images decode straight into the input tensor; the others into the raw buffers, a chunk of raw_slots at
        // a time, each chunk letter-boxed by one launch (all of it stream-ordered: a raw buffer is reused only behind its reader)
        for (int i0 = 0; i0 < n;) {
            std::vector<uint8_t *> dst;
            std::vector<LbItem> lb;
            int i1 = i0, used = 0;
            for (; i1 < n; i1++) {
                const bool direct = w[i1] == Wn && hg[i1] == Hn;
                if (!direct && used == h->raw_slots) break;
                dst.push_back(direct ? h->d_input + (size_t)i1 * img_bytes : h->d_raw + (size_t)used * h->raw_bytes);
                if (!direct) {
                    lb.emplace_back();
                    letterbox_fill(lb.back(), dst.back(), w[i1], hg[i1], h->d_input + (size_t)i1 * img_bytes, Wn, Hn, 0, area);
                    used++;
                }
            }
            if ((rc = jpeg_decode(h, jpegs + i0, jpeg_bytes + i0, i1 - i0, dst.data(), w.data() + i0, hg.data() + i0, h->stream))) return rc;
            if (!lb.empty()) CK(launch_letterbox_batch(lb.data(), (int)lb.size(), Wn, Hn, h->stream));
            i0 = i1;
        }
        set_params(h, thr, nms);
        forward_graph(h, n);
        fetch_results(h, n, out_faces, out_counts, out_idx, nullptr);
    } catch (const CudaFail &f) { return fail_cuda(h, f); }
    return RF_OK;
}

int rf_decode_jpeg(rf_handle h, const uint8_t *jpeg, size_t bytes, uint8_t *out_bgr, size_t out_capacity, int *width, int *height) {
    if (!h) return RF_ERR_INVALID_ARG;
    if (!jpeg || !bytes || !width || !height) return fail(h, RF_ERR_INVALID_ARG, "rf_decode_jpeg: NULL argument");
    try {
        CK(cudaSetDevice(h->device));
        switch_ctx(h, 0);
        int rc = jpeg_info(h, jpeg, bytes, width, height);
        if (rc) return rc;
        if (!out_bgr) return RF_OK;                                    // size query
        const size_t need = (size_t)*width * *height * 3;
        if (need > out_capacity) return fail(h, RF_ERR_CAPACITY, fmt("rf_decode_jpeg: %dx%d needs %zu bytes, the buffer has %zu", *width, *height, need, out_capacity));
        if (*width > h->cfg.max_image_w || *height > h->cfg.max_image_h)
            return fail(h, RF_ERR_CAPACITY, fmt("JPEG is %dx%d, larger than max_image %dx%d", *width, *height, h->cfg.max_image_w, h->cfg.max_image_h));
        uint8_t *dst = h->d_raw;
        if ((rc = jpeg_decode(h, &jpeg, &bytes, 1, &dst, width, height, h->stream))) return rc;
        CK(cudaMemcpyAsync(out_bgr, h->d_raw, need, cudaMemcpyDeviceToHost, h->stream));
        CK(cudaStreamSynchronize(h->stream));
    } catch (const CudaFail &f) { return fail_cuda(h, f); }
    return RF_OK;
}

const char *rf_jpeg_backend(rf_handle h) { return h ? jpeg_backend(h) : "none"; }

static void ensure_slots(rf_handle h) {
    if (h->copy_stream) return;
    const size_t in_bytes = (size_t)h->cfg.max_batch * h->cfg.net_h * h->cfg.net_w * 3;
    CK(cudaStreamCreateWithFlags(&h->copy_stream, cudaStreamNonBlocking));
    for (auto &sl : h->slots) {
        CK(cudaMalloc(&sl.d_in, in_bytes));
        CK(cudaHostAlloc(&sl.h_in, in_bytes, cudaHostAllocDefault));
        CK(cudaHostAlloc(&sl.h_dets, sizeof(rf_det) * (size_t)h->cfg.max_batch * h->cfg.max_faces, cudaHostAllocDefault));
        CK(cudaHostAlloc(&sl.h_counts, sizeof(int) * h->cfg.max_batch, cudaHostAllocDefault));
        CK(cudaEventCreateWithFlags(&sl.ev_h2d, cudaEventDisableTiming));
        CK(cudaEventCreateWithFlags(&sl.ev_done, cudaEventDisableTiming));
    }
}

static int submit_impl(rf_handle h, const uint8_t *const *imgs, int n, float thr, float nms, int *ticket, bool gather) {
    int rc = check_n(h, n);
    if (rc) return rc;
    if (!imgs || !ticket || n == 0) return fail(h, RF_ERR_INVALID_ARG, "rf_submit_batch: NULL argument or empty batch");
    if (gather && !h->comm.ready) return fail(h, RF_ERR_INVALID_ARG, "rf_submit_batch_allgather: call rf_comm_init first");
    const size_t img_bytes = (size_t)h->cfg.net_h * h->cfg.net_w * 3;
    try {
        CK(cudaSetDevice(h->device));
        ensure_slots(h);
        switch_ctx(h, (int)(h->submit_seq % (unsigned)h->nctx));
        rf_handle_s::Slot &sl = h->slots[h->submit_seq % RF_PIPELINE_DEPTH];
        if (sl.busy) return fail(h, RF_ERR_CAPACITY, "rf_submit_batch: RF_PIPELINE_DEPTH batches already in flight; collect one first");
        // H2D on the copy stream: adjacent sources collapse into one copy
        const uint8_t *run_src = nullptr;
        int run_start = -1, run_len = 0;
        auto flush = [&]() {
            if (run_start < 0) return;
            CK(cudaMemcpyAsync(sl.d_in + (size_t)run_start * img_bytes, run_src, (size_t)run_len * img_bytes, cudaMemcpyHostToDevice,
                               h->copy_stream));
            run_start = -1;
        };
        for (int i = 0; i < n; i++) {
            if (!imgs[i]) return fail(h, RF_ERR_INVALID_ARG, fmt("rf_submit_batch: image %d is NULL", i));
            const uint8_t *src = imgs[i];
            cudaPointerAttributes at{};
            bool pinned = cudaPointerGetAttributes(&at, src) == cudaSuccess && at.type == cudaMemoryTypeHost;
            if (!pinned) {
                cudaGetLastError();
                memcpy(sl.h_in + (size_t)i * img_bytes, src, img_bytes);   // slot is free: its previous H2D completed before collect
                src = sl.h_in + (size_t)i * img_bytes;
            }
            if (run_start >= 0 && src == run_src + (size_t)run_len * img_bytes) run_len++;
            else { flush(); run_start = i; run_src = src; run_len = 1; }
        }
        flush();
        CK(cudaEventRecord(sl.ev_h2d, h->copy_stream));
        CK(cudaStreamWaitEvent(h->stream, sl.ev_h2d, 0));
        if (h->param_seq && h->param_seq % rf_handle_s::kParamSlots == 0) CK(cudaStreamSynchronize(h->stream));
        const unsigned seq = gather ? ++h->comm.seq : 0u;
        set_params(h, thr, nms, sl.d_in, seq);
        forward_graph(h, n);
        if (gather) {
            // results of ALL ranks: wait for every rank's flags of this step, then read this rank's window slot
            Comm::Slot &cs = h->comm.slots[h->submit_seq % RF_PIPELINE_DEPTH];
            const size_t nimg = (size_t)h->comm.world * h->cfg.max_batch;
            if (!cs.h_dets) {
                CK(cudaHostAlloc(&cs.h_dets, sizeof(rf_det) * nimg * h->cfg.max_faces, cudaHostAllocDefault));
                CK(cudaHostAlloc(&cs.h_counts, sizeof(int) * nimg, cudaHostAllocDefault));
            }
            const unsigned slot = seq % (unsigned)h->comm.ring;
            const size_t img0 = (size_t)slot * nimg;
            CK(cudaMemcpyAsync(cs.h_counts, h->pb.comm.counts[h->comm.rank] + img0, sizeof(int) * nimg, cudaMemcpyDeviceToHost, h->stream));
            CK(cudaMemcpyAsync(cs.h_dets, h->pb.comm.dets[h->comm.rank] + img0 * h->cfg.max_faces, sizeof(rf_det) * nimg * h->cfg.max_faces, cudaMemcpyDeviceToHost,
                               h->stream));
            CK(cudaMemcpyAsync(h->comm.h_err, h->comm.d_err, 4, cudaMemcpyDeviceToHost, h->stream));
        } else {
            CK(cudaMemcpyAsync(sl.h_counts, h->pb.out_counts, sizeof(int) * n, cudaMemcpyDeviceToHost, h->stream));
            CK(cudaMemcpyAsync(sl.h_dets, h->pb.out_dets, sizeof(rf_det) * (size_t)n * h->cfg.max_faces, cudaMemcpyDeviceToHost, h->stream));
        }
        CK(cudaEventRecord(sl.ev_done, h->stream));
        sl.n = n;
        sl.busy = true;
        sl.gather = gather;
        *ticket = (int)h->submit_seq++;
    } catch (const CudaFail &f) { return fail_cuda(h, f); }
    return RF_OK;
}

int rf_submit_batch(rf_handle h, const uint8_t *const *imgs, int n, float thr, float nms, int *ticket) {
    return submit_impl(h, imgs, n, thr, nms, ticket, false);
}
int rf_submit_batch_allgather(rf_handle h, const uint8_t *const *imgs, int n, float thr, float nms, int *ticket) {
    return submit_impl(h, imgs, n, thr, nms, ticket, true);
}

static int collect_impl(rf_handle h, int ticket, rf_face *out_faces, int *out_counts, int32_t *out_idx, bool gather) {
    if (!h) return RF_ERR_INVALID_ARG;
    if ((unsigned)ticket != h->collect_seq) return fail(h, RF_ERR_INVALID_ARG, fmt("rf_collect_batch: ticket %d out of order (next is %u)", ticket, h->collect_seq));
    rf_handle_s::Slot &sl = h->slots[h->collect_seq % RF_PIPELINE_DEPTH];
    if (!sl.busy) return fail(h, RF_ERR_INVALID_ARG, "rf_collect_batch: nothing submitted under this ticket");
    if (sl.gather != gather) return fail(h, RF_ERR_INVALID_ARG, "rf_collect_batch: ticket was submitted with the other (all-gather / local) entry point");
    try {
        CK(cudaSetDevice(h->device));
        CK(cudaEventSynchronize(sl.ev_done));
    } catch (const CudaFail &f) { return fail_cuda(h, f); }
    const int mf = h->cfg.max_faces;
    const rf_det *dets = sl.h_dets;
    const int *counts = sl.h_counts;
    int nimg = sl.n;
    if (gather) {
        Comm::Slot &cs = h->comm.slots[h->collect_seq % RF_PIPELINE_DEPTH];
        dets = cs.h_dets; counts = cs.h_counts;
        if (*h->comm.h_err) {
            sl.busy = false;
            h->collect_seq++;
            return fail(h, RF_ERR_CUDA, fmt("multi-GPU exchange: rank %u never delivered its records of this step", *h->comm.h_err - 1));
        }
        // rank r's image i at r * max_batch + i; images beyond a rank's n are reported empty
        for (int r = 0; r < h->comm.world; r++)
            for (int i = sl.n; i < h->cfg.max_batch; i++)
                if (out_counts) out_counts[r * h->cfg.max_batch + i] = 0;
        for (int r = 0; r < h->comm.world; r++)
            for (int i = 0; i < sl.n; i++) {
                const size_t g = (size_t)r * h->cfg.max_batch + i;
                const int k = std::min(counts[g], mf);
                if (out_counts) out_counts[g] = k;
                for (int j = 0; j < k; j++) {
                    const rf_det &d = dets[g * mf + j];
                    if (out_faces) out_faces[g * mf + j] = d.face;
                    if (out_idx) out_idx[g * mf + j] = d.anchor_index;
                }
            }
        sl.busy = false;
        h->collect_seq++;
        return RF_OK;
    }
    for (int i = 0; i < nimg; i++) {
        const int k = counts[i];
        if (out_counts) out_counts[i] = k;
        for (int j = 0; j < k; j++) {
            const rf_det &d = dets[(size_t)i * mf + j];
            if (out_faces) out_faces[(size_t)i * mf + j] = d.face;
            if (out_idx) out_idx[(size_t)i * mf + j] = d.anchor_index;
        }
    }
    sl.busy = false;
    h->collect_seq++;
    return RF_OK;
}

int rf_collect_batch(rf_handle h, int ticket, rf_face *out_faces, int *out_counts, int32_t *out_idx) {
    return collect_impl(h, ticket, out_faces, out_counts, out_idx, false);
}
int rf_collect_batch_allgather(rf_handle h, int ticket, rf_face *out_faces, int *out_counts, int32_t *out_idx) {
    return collect_impl(h, ticket, out_faces, out_counts, out_idx, true);
}
int rf_detect_batch_allgather(rf_handle h, const uint8_t *const *imgs, int n, float thr, float nms, rf_face *out_faces, int *out_counts, int32_t *out_idx) {
    int t = 0;
    int rc = rf_submit_batch_allgather(h, imgs, n, thr, nms, &t);
    if (rc) return rc;
    return rf_collect_batch_allgather(h, t, out_faces, out_counts, out_idx);
}

static void ensure_merge_buffers(rf_handle h) {
    PostBuffers &pb = h->pb_merge;
    if (pb.cand_keys) return;
    const int A = h->cfg.max_batch * h->cfg.max_faces;       // every view may contribute max_faces candidates
    int ap2 = 1;
    while (ap2 < A) ap2 <<= 1;
    pb.anchors_per_image = A; pb.anchors_pow2 = ap2; pb.max_faces = h->cfg.max_faces; pb.max_batch = 1;
    CK(cudaMalloc(&pb.cand_keys, sizeof(unsigned long long) * (size_t)A));
    CK(cudaMalloc(&pb.cand_recs, sizeof(rf_det) * (size_t)A));
    CK(cudaMalloc(&pb.cand_count, sizeof(int)));
    CK(cudaMemset(pb.cand_count, 0, sizeof(int)));
    CK(cudaMalloc(&pb.sort_scratch, sizeof(unsigned long long) * (size_t)ap2));
    CK(cudaMalloc(&pb.flag_scratch, (size_t)ap2));
    CK(cudaMalloc(&pb.out_dets, sizeof(rf_det) * (size_t)pb.max_faces));
    CK(cudaMalloc(&pb.out_counts, sizeof(int)));
    CK(cudaMalloc(&pb.out_total_kept, sizeof(int)));
    CK(cudaMemset(pb.out_counts, 0, sizeof(int)));
}

int rf_detect_views(rf_handle h, const uint8_t *bgr, int width, int height, int row_stride, const rf_view *views, int nviews, float thr,
                    float nms, rf_face *out_faces, int *out_count, int32_t *out_view_of, float *out_view_scales) {
    if (!h || !bgr || !views || !out_count || width <= 0 || height <= 0) return fail(h, RF_ERR_INVALID_ARG, "rf_detect_views: bad arguments");
    if (nviews < 1 || nviews > RF_MAX_VIEWS || nviews > h->cfg.max_batch)
        return fail(h, RF_ERR_CAPACITY, fmt("rf_detect_views: %d views, limit min(RF_MAX_VIEWS = %d, max_batch = %d)", nviews, RF_MAX_VIEWS, h->cfg.max_batch));
    if (width > h->cfg.max_image_w || height > h->cfg.max_image_h) return fail(h, RF_ERR_CAPACITY, "rf_detect_views: image larger than max_image");
    for (int v = 0; v < nviews; v++)
        if (!(views[v].shrink > 0.f && views[v].shrink <= 1.f)) return fail(h, RF_ERR_INVALID_ARG, fmt("rf_detect_views: view %d: shrink must be in (0, 1]", v));
    static_assert(RF_MAX_VIEWS == RF_MAX_VIEWS_DEV, "view capacity of the merge kernel");
    const int Hn = h->cfg.net_h, Wn = h->cfg.net_w, mf = h->cfg.max_faces;
    const size_t img_bytes = (size_t)Hn * Wn * 3;
    const int rs = row_stride ? row_stride : width * 3;
    try {
        CK(cudaSetDevice(h->device));
        switch_ctx(h, 0);
        ensure_merge_buffers(h);
        const uint8_t *d_src = upload_raw(h, bgr, width, height, rs);
        ViewSet vs{};
        vs.nviews = nviews;
        vs.img_w_minus1 = (float)(width - 1);
        const int area = (h->cfg.flags & RF_FLAG_NPP_RESIZE) ? 1 : 0;
        std::vector<LbItem> lb(nviews);
        for (int v = 0; v < nviews; v++) {
            const int bw = std::max(1, (int)(Wn * views[v].shrink)), bh = std::max(1, (int)(Hn * views[v].shrink));
            vs.flip[v] = views[v].flip ? 1 : 0;
            vs.scale[v] = letterbox_fill(lb[v], d_src, width, height, h->d_input + (size_t)v * img_bytes, bw, bh, vs.flip[v], area);
            if (out_view_scales) out_view_scales[v] = vs.scale[v];
        }
        CK(launch_letterbox_batch(lb.data(), nviews, Wn, Hn, h->stream));     // all views of the image: one launch
        set_params(h, thr, nms);
        forward_graph(h, nviews);
        launch_merge_views(h->pb, vs, h->pb_merge, h->stream);
        launch_nms(1, h->d_params, h->pb_merge, h->stream);
        CK(cudaMemcpyAsync(h->h_counts, h->pb_merge.out_counts, sizeof(int), cudaMemcpyDeviceToHost, h->stream));
        CK(cudaMemcpyAsync(h->h_dets, h->pb_merge.out_dets, sizeof(rf_det) * (size_t)mf, cudaMemcpyDeviceToHost, h->stream));
        CK(cudaStreamSynchronize(h->stream));
        const int k = h->h_counts[0];
        *out_count = k;
        for (int j = 0; j < k; j++) {
            if (out_faces) out_faces[j] = h->h_dets[j].face;
            if (out_view_of) out_view_of[j] = h->h_dets[j].anchor_index / mf;
        }
    } catch (const CudaFail &f) { return fail_cuda(h, f); }
    return RF_OK;
}

int rf_preprocess(rf_handle h, const uint8_t *bgr, int width, int height, int row_stride, uint8_t *out) {
    if (!h || !bgr || !out || width <= 0 || height <= 0) return fail(h, RF_ERR_INVALID_ARG, "rf_preprocess: bad arguments");
    if (width > h->cfg.max_image_w || height > h->cfg.max_image_h) return fail(h, RF_ERR_CAPACITY, "rf_preprocess: image larger than max_image");
    const int Hn = h->cfg.net_h, Wn = h->cfg.net_w;
    const int rs = row_stride ? row_stride : width * 3;
    try {
        CK(cudaSetDevice(h->device));
        switch_ctx(h, 0);
        const uint8_t *d_src = upload_raw(h, bgr, width, height, rs);
        LbItem it;
        letterbox_fill(it, d_src, width, height, h->d_input, Wn, Hn, 0, (h->cfg.flags & RF_FLAG_NPP_RESIZE) ? 1 : 0);
        CK(launch_letterbox_batch(&it, 1, Wn, Hn, h->stream));
        CK(cudaMemcpyAsync(h->h_input, h->d_input, (size_t)Hn * Wn * 3, cudaMemcpyDeviceToHost, h->stream));
        CK(cudaStreamSynchronize(h->stream));
        memcpy(out, h->h_input, (size_t)Hn * Wn * 3);
    } catch (const CudaFail &f) { return fail_cuda(h, f); }
    return RF_OK;
}

static void ensure_blobs(rf_handle h) {
    if (h->d_blobs[0]) return;
    for (int i = 0; i < 9; i++) CK(cudaMalloc(&h->d_blobs[i], sizeof(float) * h->blob_elems[i] * h->cfg.max_batch));
}

int rf_forward_heads(rf_handle h, const uint8_t *bgr, int n, float *const heads_out[9]) {
    int rc = check_n(h, n);
    if (rc) return rc;
    if (n == 0) return RF_OK;
    if (!bgr || !heads_out) return fail(h, RF_ERR_INVALID_ARG, "rf_forward_heads: NULL argument");
    try {
        CK(cudaSetDevice(h->device));
        switch_ctx(h, 0);
        ensure_blobs(h);
        const size_t bytes = (size_t)n * h->cfg.net_h * h->cfg.net_w * 3;
        CK(cudaStreamSynchronize(h->stream));
        memcpy(h->h_input, bgr, bytes);
        CK(cudaMemcpyAsync(h->d_input, h->h_input, bytes, cudaMemcpyHostToDevice, h->stream));
        set_params(h, h->cur_thr, h->cur_nms);
        h->blobs_in_plan = true;
        try { run_steps(h, n, h->stream); } catch (...) { h->blobs_in_plan = false; throw; }
        h->blobs_in_plan = false;
        CK(cudaGetLastError());
        for (int i = 0; i < 9; i++)
            CK(cudaMemcpyAsync(heads_out[i], h->d_blobs[i], sizeof(float) * h->blob_elems[i] * n, cudaMemcpyDeviceToHost, h->stream));
        CK(cudaStreamSynchronize(h->stream));
    } catch (const CudaFail &f) { return fail_cuda(h, f); }
    return RF_OK;
}

int rf_postprocess(rf_handle h, const float *const heads[9], int n, float thr, float nms, rf_face *out_faces, int *out_counts,
                   int32_t *out_idx, int *out_ncand) {
    int rc = check_n(h, n);
    if (rc) return rc;
    if (n == 0) return RF_OK;
    if (!heads) return fail(h, RF_ERR_INVALID_ARG, "rf_postprocess: NULL heads");
    try {
        CK(cudaSetDevice(h->device));
        switch_ctx(h, 0);
        ensure_blobs(h);
        for (int i = 0; i < 9; i++)
            CK(cudaMemcpyAsync(h->d_blobs[i], heads[i], sizeof(float) * h->blob_elems[i] * n, cudaMemcpyHostToDevice, h->stream));
        set_params(h, thr, nms);
        launch_blob_decode(h->d_blobs, h->lv, n, h->cfg.net_w, h->cfg.net_h, h->d_params, h->pb, h->stream);
        if (out_ncand) CK(cudaMemcpyAsync(h->h_counts + h->cfg.max_batch, h->pb.cand_count, sizeof(int) * n, cudaMemcpyDeviceToHost, h->stream));
        launch_nms(n, h->d_params, h->pb, h->stream);
        CK(cudaGetLastError());
        fetch_results(h, n, out_faces, out_counts, out_idx, nullptr);
        if (out_ncand) for (int i = 0; i < n; i++) out_ncand[i] = h->h_counts[h->cfg.max_batch + i];
    } catch (const CudaFail &f) { return fail_cuda(h, f); }
    return RF_OK;
}

// Debug / parity: any materialised activation by its Caffe top name, as NCHW float32.
int rf_debug_get_tensor(rf_handle h, const char *name, int n, float *out_nchw, int *c, int *hh, int *ww) {
    int rc = check_n(h, n);
    if (rc) return rc;
    auto it = h->tensor_by_name.find(name ? name : "");
    if (it == h->tensor_by_name.end()) return fail(h, RF_ERR_INVALID_ARG, fmt("unknown tensor '%s'", name ? name : "(null)"));
    const TensorInfo &t = h->tensors[it->second];
    if (c) *c = t.c;
    if (hh) *hh = t.h;
    if (ww) *ww = t.w;
    if (!out_nchw) return RF_OK;
    try {
        CK(cudaSetDevice(h->device));
        switch_ctx(h, 0);
        CK(cudaStreamSynchronize(h->stream));
        size_t elems = (size_t)n * t.h * t.w * t.c;
        std::vector<unsigned char> host(elems * h->elem);
        CK(cudaMemcpy(host.data(), h->tptr(it->second), host.size(), cudaMemcpyDeviceToHost));
        for (int b = 0; b < n; b++)
            for (int y = 0; y < t.h; y++)
                for (int x = 0; x < t.w; x++)
                    for (int ch = 0; ch < t.c; ch++) {
                        size_t src = (((size_t)b * t.h + y) * t.w + x) * t.c + ch;
                        float v = h->elem == 4 ? reinterpret_cast<float *>(host.data())[src]
                                : h->elem == 2 ? __half2float(reinterpret_cast<__half *>(host.data())[src])
                                               : (float)reinterpret_cast<int8_t *>(host.data())[src];   // INT8: raw quantised values
                        out_nchw[(((size_t)b * t.c + ch) * t.h + y) * t.w + x] = v;
                    }
    } catch (const CudaFail &f) { return fail_cuda(h, f); }
    return RF_OK;
}

// Re-places activations without buffer reuse so that rf_debug_get_tensor sees every tensor of
// the last forward (debug only; call before the first forward).
int rf_debug_keep_all(rf_handle h) {
    if (!h) return RF_ERR_INVALID_ARG;
    try {
        CK(cudaSetDevice(h->device));
        for (auto &t : h->tensors) { t.first = -1; t.last = -1; }
        place_tensors(h, true);
        for (int c = 0; c < h->nctx; c++) {
            switch_ctx(h, c);
            CK(cudaStreamSynchronize(h->stream));
            for (auto &g : h->graphs) cudaGraphExecDestroy(g.second);
            h->graphs.clear();
            CK(cudaFree(h->arena));
            h->arena = nullptr;
            CK(cudaMalloc(&h->arena, h->arena_bytes));
        }
        switch_ctx(h, 0);
    } catch (const CudaFail &f) { return fail_cuda(h, f); }
    return RF_OK;
}

// INT8 entropy calibration (SURVEY.md 8f-3; replaces INT8-Calibration-Tool/calibrationtable.cpp:399-583).  `h` must be an
// RF_PREC_FP32 handle (its SIMT plan materialises every tensor the INT8 plan quantises, including the depthwise outputs
// and the FPN sums).  Two passes over the n network-sized images: absmax, then 2048-bin histograms; then the KL threshold
// search per tensor on the host; the table is written in the reference's TensorRT cache format.
int rf_calibrate_int8(rf_handle h, const uint8_t *bgr_net_sized, int n_images, const char *out_table_path) {
    if (!h || !bgr_net_sized || n_images <= 0 || !out_table_path) return fail(h, RF_ERR_INVALID_ARG, "rf_calibrate_int8: bad arguments");
    if (h->cfg.precision != RF_PREC_FP32) return fail(h, RF_ERR_UNSUPPORTED, "rf_calibrate_int8: create the handle with RF_PREC_FP32 (every tensor must be materialised)");
    const size_t img_bytes = (size_t)h->cfg.net_h * h->cfg.net_w * 3;
    const int T = (int)h->tensors.size();
    float *d_max = nullptr;
    unsigned *d_hist = nullptr;
    try {
        CK(cudaSetDevice(h->device));
        int rc = rf_debug_keep_all(h);
        if (rc) return rc;
        switch_ctx(h, 0);
        CK(cudaMalloc(&d_max, sizeof(float) * T));
        CK(cudaMalloc(&d_hist, sizeof(unsigned) * (size_t)T * CALIB_BINS));
        CK(cudaMemsetAsync(d_max, 0, sizeof(float) * T, h->stream));
        CK(cudaMemsetAsync(d_hist, 0, sizeof(unsigned) * (size_t)T * CALIB_BINS, h->stream));
        std::vector<float> hmax(T, 0.f);
        for (int pass = 0; pass < 2; pass++) {
            for (int i0 = 0; i0 < n_images; i0 += h->cfg.max_batch) {
                const int n = std::min(h->cfg.max_batch, n_images - i0);
                CK(cudaStreamSynchronize(h->stream));
                memcpy(h->h_input, bgr_net_sized + (size_t)i0 * img_bytes, (size_t)n * img_bytes);
                CK(cudaMemcpyAsync(h->d_input, h->h_input, (size_t)n * img_bytes, cudaMemcpyHostToDevice, h->stream));
                set_params(h, h->cur_thr, h->cur_nms);
                run_steps(h, n, h->stream, false);
                for (int t = 0; t < T; t++) {
                    const TensorInfo &ti = h->tensors[t];
                    const size_t elems = (size_t)n * ti.h * ti.w * ti.c;
                    const float *x = reinterpret_cast<const float *>(h->tptr(t));
                    if (pass == 0) launch_absmax<float>(x, elems, d_max + t, h->stream);
                    else if (hmax[t] > 0.f) launch_hist<float>(x, elems, (float)CALIB_BINS / hmax[t], d_hist + (size_t)t * CALIB_BINS, h->stream);
                }
                CK(cudaGetLastError());
            }
            if (pass == 0) {
                CK(cudaMemcpyAsync(hmax.data(), d_max, sizeof(float) * T, cudaMemcpyDeviceToHost, h->stream));
                CK(cudaStreamSynchronize(h->stream));
            }
        }
        std::vector<unsigned> hist((size_t)T * CALIB_BINS);
        CK(cudaMemcpyAsync(hist.data(), d_hist, sizeof(unsigned) * hist.size(), cudaMemcpyDeviceToHost, h->stream));
        CK(cudaStreamSynchronize(h->stream));
        cudaFree(d_max); cudaFree(d_hist);
        d_max = nullptr; d_hist = nullptr;
        std::vector<std::pair<std::string, float>> scales;
        scales.emplace_back("data", 255.0f / 127.0f);          // u8 input range; the engine consumes the u8 image directly
        for (int t = 0; t < T; t++) {
            if (hmax[t] <= 0.f) { scales.emplace_back(h->tensors[t].name, 1.0f / 127.0f); continue; }
            const double bins = kl_threshold_bins(hist.data() + (size_t)t * CALIB_BINS);
            const double thr = bins * (double)hmax[t] / CALIB_BINS;
            scales.emplace_back(h->tensors[t].name, (float)(thr / 127.0));
        }
        std::string err;
        if (!write_int8_table(out_table_path, scales, err)) return fail(h, RF_ERR_IO, err);
    } catch (const CudaFail &f) {
        cudaFree(d_max); cudaFree(d_hist);
        return fail_cuda(h, f);
    }
    return RF_OK;
}

// Host-only: the KL threshold search on a caller-supplied histogram (for CPU-side tests of the calibrator).
double rf_kl_threshold_bins(const unsigned *hist, int bins, int levels) { return kl_threshold_bins(hist, bins, levels); }

// Host-only (no GPU needed): folded FP32 weights/bias of one convolution as the engine will hold
// them (BatchNorm + Scale + bias folded).  dims = {cout, cin/groups, k, k}.  Lets CPU-only tests
// check the model front end against the oracle's fold.
int rf_cache_status(rf_handle h) { return h ? h->cache_status : RF_ERR_INVALID_ARG; }

int rf_network_config(const char *network, int *num_levels, int strides[3], int scales[6], float ratios[2], int *num_ratios) {
    if (!network) return fail(nullptr, RF_ERR_INVALID_ARG, "rf_network_config: NULL network");
    NetworkConfig nc;
    std::string err;
    const bool ok = network_config(network, nc, err);
    if (num_ratios) *num_ratios = (int)nc.ratios.size();
    if (ratios) for (size_t i = 0; i < nc.ratios.size() && i < 2; i++) ratios[i] = nc.ratios[i];
    if (!ok) return fail(nullptr, RF_ERR_UNSUPPORTED, err);
    if (num_levels) *num_levels = (int)nc.strides.size();
    for (size_t l = 0; l < nc.strides.size() && l < 3; l++) {
        if (strides) strides[l] = nc.strides[l];
        if (scales) { scales[2 * l] = nc.scales[l][0]; scales[2 * l + 1] = nc.scales[l][1]; }
    }
    return RF_OK;
}

int rf_model_load(const char *caffemodel_path, const char *prototxt_path, const char *cache_path, int *cache_status, int input_dims[4],
                  const char *layer, float *w, int wcap, float *b, int bcap, int dims[4]) {
    if (!caffemodel_path) return fail(nullptr, RF_ERR_INVALID_ARG, "rf_model_load: NULL caffemodel_path");
    Model m;
    NetGraph g;
    std::string err;
    int st = RF_OK, cs = CACHE_NONE;
    if (!load_model(caffemodel_path, prototxt_path ? prototxt_path : "", cache_path ? cache_path : "", m, &g, &cs, err, st)) return fail(nullptr, st, err);
    if (cache_status) *cache_status = cs;
    if (input_dims) for (int k = 0; k < 4; k++) input_dims[k] = g.input_dims[k];
    if (!layer) return RF_OK;
    auto it = m.convs.find(layer);
    if (it == m.convs.end()) return fail(nullptr, RF_ERR_INVALID_ARG, std::string("no convolution '") + layer + "'");
    const FoldedConv &c = it->second;
    if (dims) { dims[0] = c.cout; dims[1] = c.cin / c.groups; dims[2] = c.k; dims[3] = c.k; }
    if (w) { if ((size_t)wcap < c.w.size()) return fail(nullptr, RF_ERR_CAPACITY, "w buffer too small"); memcpy(w, c.w.data(), c.w.size() * 4); }
    if (b) { if ((size_t)bcap < c.b.size()) return fail(nullptr, RF_ERR_CAPACITY, "b buffer too small"); memcpy(b, c.b.data(), c.b.size() * 4); }
    return RF_OK;
}

int rf_model_inspect(const char *caffemodel_path, const char *layer, float *w, int wcap, float *b, int bcap, int dims[4]) {
    if (!caffemodel_path || !layer) return fail(nullptr, RF_ERR_INVALID_ARG, "rf_model_inspect: NULL argument");
    std::vector<RawLayer> layers;
    std::string err;
    bool io = false;
    Model m;
    if (!read_caffemodel(caffemodel_path, layers, err, io)) return fail(nullptr, io ? RF_ERR_IO : RF_ERR_MODEL, err);
    if (!build_mnet_model(layers, m, err)) return fail(nullptr, RF_ERR_MODEL, err);
    auto it = m.convs.find(layer);
    if (it == m.convs.end()) return fail(nullptr, RF_ERR_INVALID_ARG, std::string("no convolution '") + layer + "'");
    const FoldedConv &c = it->second;
    if (dims) { dims[0] = c.cout; dims[1] = c.cin / c.groups; dims[2] = c.k; dims[3] = c.k; }
    if (w) { if ((size_t)wcap < c.w.size()) return fail(nullptr, RF_ERR_CAPACITY, "w buffer too small"); memcpy(w, c.w.data(), c.w.size() * 4); }
    if (b) { if ((size_t)bcap < c.b.size()) return fail(nullptr, RF_ERR_CAPACITY, "b buffer too small"); memcpy(b, c.b.data(), c.b.size() * 4); }
    return RF_OK;
}

// Host-only (works without a GPU): builds the layer plan rf_create would build for `cfg` and writes one line per kernel
// launch of a forward (and, for tile chains, their geometry and shared-memory / TMEM budget) into `out`.
int rf_plan_describe(const rf_config *cfg, char *out, int cap) {
    if (!cfg || !cfg->caffemodel_path || !out || cap <= 0) return fail(nullptr, RF_ERR_INVALID_ARG, "rf_plan_describe: bad arguments");
    if (cfg->net_w <= 0 || cfg->net_h <= 0 || cfg->net_w % 32 || cfg->net_h % 32 || cfg->max_batch <= 0)
        return fail(nullptr, RF_ERR_INVALID_ARG, "rf_plan_describe: bad network size / batch");
    std::unique_ptr<rf_handle_s> H(new rf_handle_s);
    rf_handle h = H.get();
    h->cfg = *cfg;
    if (h->cfg.max_faces <= 0) h->cfg.max_faces = 256;
    h->elem = cfg->precision == RF_PREC_FP32 ? 4 : (cfg->precision == RF_PREC_FP16 ? 2 : 1);
    std::vector<RawLayer> layers;
    std::string err;
    bool io = false;
    if (!read_caffemodel(cfg->caffemodel_path, layers, err, io)) return fail(nullptr, io ? RF_ERR_IO : RF_ERR_MODEL, err);
    if (!build_mnet_model(layers, h->model, err)) return fail(nullptr, RF_ERR_MODEL, err);
    if (cfg->int8_table_path && !read_int8_table(cfg->int8_table_path, h->int8_scales, err)) return fail(nullptr, RF_ERR_IO, err);
    try {
        h->use_tc = cfg->precision == RF_PREC_INT8 || (cfg->precision == RF_PREC_FP16 && !(cfg->flags & RF_FLAG_NO_TENSORCORE));
        if (cfg->precision == RF_PREC_INT8) build_plan_i8(h);
        else if (cfg->precision == RF_PREC_FP32) build_plan<float>(h);
        else if (h->use_tc && !(cfg->flags & RF_FLAG_LEGACY_TC)) build_plan_tiles(h);
        else build_plan<__half>(h);
        link_steps(h);
        place_tensors(h, false);
    } catch (const CudaFail &f) { return fail_cuda(nullptr, f); }
    catch (const PlanFail &f) { return fail(nullptr, f.status, f.msg); }
    std::string text = fmt("%d launches per forward, activation arena %zu bytes per batch of %d\n", (int)h->steps.size(), h->arena_bytes, cfg->max_batch);
    for (auto &st : h->steps) text += fmt("step lane %d: %s\n", st.lane, st.name.c_str());
    text += describe_chains(h);
    snprintf(out, (size_t)cap, "%s", text.c_str());
    return (int)h->steps.size();
}

int rf_profile_layers(rf_handle h, int n, int iters, char (*names)[64], float *ms, double *bytes, double *flops, int cap) {
    int rc = check_n(h, n);
    if (rc) return rc;
    if (n == 0 || iters <= 0) return fail(h, RF_ERR_INVALID_ARG, "rf_profile_layers: n and iters must be positive");
    int cnt = 0;
    try {
        CK(cudaSetDevice(h->device));
        switch_ctx(h, 0);
        set_params(h, h->cur_thr, h->cur_nms);
        run_steps(h, n, h->stream, false);  // warm everything once (also leaves consistent inputs for every step)
        CK(cudaStreamSynchronize(h->stream));
        struct ProfGuard { rf_handle h; ~ProfGuard() { h->profiling = false; } } guard{h};
        h->profiling = true;
        for (size_t si = 0; si < h->steps.size(); si++) {
            auto &st = h->steps[si];
            if (cnt >= cap) break;
            if ((int)si == h->head_step + 1) {
                // sort+nms consumes the candidate list: give every timed launch a fresh one
                float acc = 0;
                for (int i = 0; i < iters; i++) {
                    h->steps[h->head_step].launch(n, h->stream);
                    CK(cudaEventRecord(h->ev0, h->stream));
                    st.launch(n, h->stream);
                    CK(cudaEventRecord(h->ev1, h->stream));
                    CK(cudaEventSynchronize(h->ev1));
                    float t = 0;
                    CK(cudaEventElapsedTime(&t, h->ev0, h->ev1));
                    acc += t;
                }
                snprintf(names[cnt], 64, "%s", st.name.c_str());
                ms[cnt] = acc / iters;
                if (bytes) bytes[cnt] = st.bytes_per_img * n;
                if (flops) flops[cnt] = st.flops_per_img * n;
                cnt++;
                continue;
            }
            st.launch(n, h->stream);
            CK(cudaEventRecord(h->ev0, h->stream));
            for (int i = 0; i < iters; i++) st.launch(n, h->stream);
            CK(cudaEventRecord(h->ev1, h->stream));
            CK(cudaEventSynchronize(h->ev1));
            float t = 0;
            CK(cudaEventElapsedTime(&t, h->ev0, h->ev1));
            snprintf(names[cnt], 64, "%s", st.name.c_str());
            ms[cnt] = t / iters;
            if (bytes) bytes[cnt] = st.bytes_per_img * n;
            if (flops) flops[cnt] = st.flops_per_img * n;
            cnt++;
        }
        CK(cudaGetLastError());
        // single steps were launched out of their forward: leave the last-block / candidate counters as a forward expects them
        CK(cudaMemsetAsync(h->pb.tile_done, 0, sizeof(int) * h->cfg.max_batch, h->stream));
        CK(cudaMemsetAsync(h->pb.cand_count, 0, sizeof(int) * h->cfg.max_batch, h->stream));
        CK(cudaStreamSynchronize(h->stream));
    } catch (const CudaFail &f) { return fail_cuda(h, f); }
    return cnt;
}

}  // extern "C"
