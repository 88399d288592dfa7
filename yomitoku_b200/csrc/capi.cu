// extern "C" surface of libytk_b200.so (declared in include/yomitoku_b200.h).
#include "../../include/yomitoku_b200.h"

#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <map>
#include <memory>
#include <mutex>
#include <tuple>

#include "crop_ops.h"
#include "dbnet_engine.h"
#include "dbnet_ops.h"
#include "dbpost_ops.h"
#include "gemm_tc.h"
#include "parseq_engine.h"
#include "rtdetr_engine.h"

// Binds the calling host thread to a device for the duration of an API call and puts the previous device back (host
// threads start on device 0, and a handle on cuda:1 must not leave "the current device" changed for the caller - PyTorch
// allocates `device="cuda"` tensors on it).
struct DevGuard {
    int prev = -1, dev = -1;
    explicit DevGuard(int d) : dev(d) {
        cudaGetDevice(&prev);
        if (prev != dev) cudaSetDevice(dev);
    }
    ~DevGuard() {
        if (prev >= 0 && prev != dev) cudaSetDevice(prev);
    }
    DevGuard(const DevGuard&) = delete;
    DevGuard& operator=(const DevGuard&) = delete;
};

struct ytk_parseq {
    ytk::ParseqModel model;
    ytk::ParseqEngine engine;
    std::mutex mu;
    int device = 0;  // the device current at create(); every later call binds the calling thread to it
};

struct ytk_dbnet {
    ytk::DbnetModel model;
    // launch plans + activation buffers per input shape (n, Hn, Wn); least recently used ones are dropped beyond
    // max_engines (YTK_DBNET_MAX_ENGINES, default 6) so that a stream of differently sized pages cannot exhaust HBM
    std::map<std::tuple<int, int, int>, std::unique_ptr<ytk::DbnetEngine>> engines;
    std::map<std::tuple<int, int, int>, unsigned long long> last_use;
    unsigned long long tick = 0;
    int max_engines = 6;
    std::mutex mu;
    int device = 0;
    int shortest = 1280, limit = 1600;
    void* stage = nullptr;  // device staging for host inputs
    size_t stage_bytes = 0;
    // The staging buffer and an engine's input / activation / probability buffers are shared by all calls on this
    // handle.  A call that leaves its output on the device returns while its kernels are still queued, so every call
    // first makes its stream wait for the previous call's last operation (recorded here), whatever stream that was on.
    cudaEvent_t last_done = nullptr;
};

static void order_after_previous(ytk_dbnet* h, cudaStream_t st) {
    if (h->last_done) cudaStreamWaitEvent(st, h->last_done, 0);
}
static void mark_done(ytk_dbnet* h, cudaStream_t st) {
    if (!h->last_done) cudaEventCreateWithFlags(&h->last_done, cudaEventDisableTiming);
    if (h->last_done) cudaEventRecord(h->last_done, st);
}

static ytk::DbnetEngine* get_engine(ytk_dbnet* h, int n, int Hn, int Wn) {
    auto key = std::make_tuple(n, Hn, Wn);
    h->last_use[key] = ++h->tick;
    auto it = h->engines.find(key);
    if (it != h->engines.end()) return it->second.get();
    while ((int)h->engines.size() >= h->max_engines && !h->engines.empty()) {
        auto victim = h->engines.begin();
        for (auto e = h->engines.begin(); e != h->engines.end(); ++e)
            if (h->last_use[e->first] < h->last_use[victim->first]) victim = e;
        cudaDeviceSynchronize();  // its last run may still be in flight on some stream
        h->last_use.erase(victim->first);
        h->engines.erase(victim);
    }
    auto e = std::make_unique<ytk::DbnetEngine>();
    if (e->build(h->model, n, Hn, Wn)) return nullptr;
    ytk::DbnetEngine* p = e.get();
    h->engines[key] = std::move(e);
    return p;
}

static int ensure_stage(ytk_dbnet* h, size_t bytes) {
    if (h->stage_bytes >= bytes) return 0;
    if (h->last_done) cudaEventSynchronize(h->last_done);  // the previous call may still be reading the old buffer
    if (h->stage) cudaFree(h->stage);
    h->stage = nullptr;
    h->stage_bytes = 0;
    if (cudaMalloc(&h->stage, bytes) != cudaSuccess) {
        ytk::set_error("cudaMalloc(%zu) for input staging failed", bytes);
        return 1;
    }
    h->stage_bytes = bytes;
    return 0;
}

static int finish_forward(ytk_dbnet* h, ytk::DbnetEngine* e, float* prob_out, int out_on_device, cudaStream_t st) {
    if (e->run(st)) return YTK_ERR;
    const size_t bytes = (size_t)e->N * e->Hn * e->Wn * sizeof(float);
    cudaError_t err = cudaMemcpyAsync(prob_out, e->prob, bytes,
                                      out_on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost, st);
    mark_done(h, st);
    if (err == cudaSuccess && !out_on_device) err = cudaStreamSynchronize(st);
    if (err != cudaSuccess) {
        ytk::set_error("DBNet output copy failed: %s", cudaGetErrorString(err));
        return YTK_ERR;
    }
    return YTK_OK;
}

extern "C" {

const char* ytk_last_error(void) { return ytk::last_error(); }
int ytk_version(void) { return 1; }
long long ytk_launch_count(void) { return ytk::launch_count(); }
void ytk_gemm_profile_begin(void) { ytk::gemm_profile_begin(); }
int ytk_gemm_profile_end(double* flops, double* ms, long long* launches) {
    return ytk::gemm_profile_end(flops, ms, launches) ? YTK_ERR : YTK_OK;
}

int ytk_op_conv2d_f16(const void* in, int N, int H, int W, int Cin, long long in_ld, const void* w, const float* bias,
                       int kh, int kw, int stride, int pad, int dil, int Cout, const void* resid, int resid_f32,
                       long long ldr, void* out, int out_f32, long long ldc, int act, int mode, void* cuda_stream) {
    ytk::ConvGeom g{N, H, W, Cin, in_ld, kh, kw, stride, pad, dil, Cout};
    ytk::Epilogue e;
    e.bias = bias;
    e.resid = resid;
    e.resid_f32 = resid_f32;
    e.ldr = ldr;
    e.out = out;
    e.out_f32 = out_f32;
    e.ldc = ldc;
    e.act = act;
    e.mode = mode;
    ytk::GemmPlan plan;
    if (ytk::conv_plan_create(&plan, in, g, w, e)) return YTK_ERR;
    return ytk::gemm_plan_launch(&plan, static_cast<cudaStream_t>(cuda_stream)) ? YTK_ERR : YTK_OK;
}

int ytk_op_linear_f16(const void* A, long long lda, int M, int K, const void* W, int N, const float* bias,
                       const void* resid, int resid_f32, long long ldr, void* out, int out_f32, long long ldc, int act,
                       void* cuda_stream) {
    ytk::Epilogue e;
    e.bias = bias;
    e.resid = resid;
    e.resid_f32 = resid_f32;
    e.ldr = ldr;
    e.out = out;
    e.out_f32 = out_f32;
    e.ldc = ldc;
    e.act = act;
    ytk::GemmPlan plan;
    if (ytk::gemm_plan_create(&plan, A, lda, M, K, W, N, e)) return YTK_ERR;
    return ytk::gemm_plan_launch(&plan, static_cast<cudaStream_t>(cuda_stream)) ? YTK_ERR : YTK_OK;
}

static_assert(sizeof(ytk_attn_seq) == sizeof(ytk::SeqDesc), "ytk_attn_seq and ytk::SeqDesc must have one layout");

int ytk_op_attention_f16(const void* Q, long long ldq, long long q_rows, const void* K, const void* V, long long ldkv,
                         long long kv_rows, void* O, long long ldo, const ytk_attn_seq* seqs_dev, int nseq, int max_q_len,
                         int heads, int head_dim, int masked, int impl, void* cuda_stream) {
    return ytk::launch_flash_attention(Q, ldq, q_rows, K, V, ldkv, kv_rows, O, ldo,
                                       reinterpret_cast<const ytk::SeqDesc*>(seqs_dev), nseq, max_q_len, heads, head_dim,
                                       masked, static_cast<cudaStream_t>(cuda_stream), impl)
               ? YTK_ERR
               : YTK_OK;
}

int ytk_op_rt_topk_f32(const float* scores_dev, int n_img, int L, int K, int* out_idx_dev, void* stream) {
    if (!scores_dev || !out_idx_dev || n_img < 1 || L < 1 || K < 1) {
        ytk::set_error("ytk_op_rt_topk_f32: bad arguments (n_img %d, L %d, K %d)", n_img, L, K);
        return YTK_ERR;
    }
    return ytk::launch_rt_topk(scores_dev, n_img, L, K, out_idx_dev, static_cast<cudaStream_t>(stream)) ? YTK_ERR : YTK_OK;
}

static_assert(sizeof(ytk_db_run) == sizeof(ytk::DbRun), "ytk_db_run and ytk::DbRun must have one layout");

int ytk_dbnet_post_front(const float* prob_dev, int n_pages, int H, int W, float thresh, void* scratch_dev,
                         long long scratch_bytes, ytk_db_run* runs_dev, int max_runs_per_page, int32_t* meta_dev,
                         void* cuda_stream) {
    if (!prob_dev || !scratch_dev || !runs_dev || !meta_dev || n_pages <= 0 || H <= 0 || W <= 0 || max_runs_per_page <= 0 ||
        (long long)H * W >= 0x7fffffffLL) {
        ytk::set_error("ytk_dbnet_post_front: bad arguments");
        return YTK_ERR;
    }
    if (scratch_bytes < ytk::dbpost_scratch_bytes(n_pages, H, W)) {
        ytk::set_error("ytk_dbnet_post_front: scratch_dev holds %lld bytes, need %lld", scratch_bytes,
                       ytk::dbpost_scratch_bytes(n_pages, H, W));
        return YTK_ERR;
    }
    cudaPointerAttributes attr;
    if (cudaPointerGetAttributes(&attr, prob_dev) != cudaSuccess || attr.type != cudaMemoryTypeDevice) {
        cudaGetLastError();
        ytk::set_error("ytk_dbnet_post_front: prob_dev is not a device pointer");
        return YTK_ERR;
    }
    DevGuard dev_guard(attr.device);
    if (ytk::launch_dbpost_front(prob_dev, n_pages, H, W, thresh, reinterpret_cast<int*>(scratch_dev),
                                 reinterpret_cast<ytk::DbRun*>(runs_dev), max_runs_per_page, meta_dev,
                                 static_cast<cudaStream_t>(cuda_stream))) {
        ytk::set_error("ytk_dbnet_post_front: kernel launch failed");
        return YTK_ERR;
    }
    return YTK_OK;
}

int ytk_dbnet_create(const ytk_tensor* tensors, int n_tensors, int shortest_size, int limit_size, ytk_dbnet** out) {
    if (!tensors || !out) {
        ytk::set_error("ytk_dbnet_create: null argument");
        return YTK_ERR;
    }
    ytk::WeightSet ws;
    for (int i = 0; i < n_tensors; ++i) {
        ytk::TensorView v;
        v.data = tensors[i].data;
        v.ndim = tensors[i].ndim;
        for (int d = 0; d < 4; ++d) v.shape[d] = d < v.ndim ? tensors[i].shape[d] : 1;
        ws.map[tensors[i].name] = v;
    }
    auto h = std::make_unique<ytk_dbnet>();
    cudaGetDevice(&h->device);
    h->shortest = shortest_size;
    h->limit = limit_size;
    if (const char* me = getenv("YTK_DBNET_MAX_ENGINES")) h->max_engines = std::max(1, atoi(me));
    if (h->model.load(ws)) return YTK_ERR;
    *out = h.release();
    return YTK_OK;
}

void ytk_dbnet_destroy(ytk_dbnet* h) {
    if (!h) return;
    DevGuard dev_guard(h->device);
    if (h->last_done) {
        cudaEventSynchronize(h->last_done);
        cudaEventDestroy(h->last_done);
    }
    if (h->stage) cudaFree(h->stage);
    delete h;
}

int ytk_dbnet_device(const ytk_dbnet* h) { return h ? h->device : -1; }
int ytk_parseq_device(const ytk_parseq* h) { return h ? h->device : -1; }

int ytk_dbnet_input_size(const ytk_dbnet* h, int H0, int W0, int* Hn, int* Wn) {
    ytk::dbnet_input_size(H0, W0, h->shortest, h->limit, Hn, Wn);
    return YTK_OK;
}

int ytk_dbnet_forward_u8(ytk_dbnet* h, const uint8_t* pages, int pages_on_device, int n_pages, int H0, int W0,
                         float* prob_out, int out_on_device, void* cuda_stream) {
    std::lock_guard<std::mutex> lk(h->mu);
    DevGuard dev_guard(h->device);  // host threads start on device 0: the handle's device is the one that counts
    cudaStream_t st = static_cast<cudaStream_t>(cuda_stream);
    int Hn, Wn;
    ytk::dbnet_input_size(H0, W0, h->shortest, h->limit, &Hn, &Wn);
    if (Hn > H0 || Wn > W0) {
        ytk::set_error("ytk_dbnet_forward_u8: page %dx%d would be upscaled to %dx%d; the fused u8 path implements "
                       "OpenCV's INTER_AREA decimation only - resize on the host and call ytk_dbnet_forward_f32",
                       H0, W0, Hn, Wn);
        return YTK_ERR;
    }
    ytk::DbnetEngine* e = get_engine(h, n_pages, Hn, Wn);
    if (!e) return YTK_ERR;
    order_after_previous(h, st);
    const uint8_t* src = pages;
    if (!pages_on_device) {
        const size_t bytes = (size_t)n_pages * H0 * W0 * 3;
        if (ensure_stage(h, bytes)) return YTK_ERR;
        if (cudaMemcpyAsync(h->stage, pages, bytes, cudaMemcpyHostToDevice, st) != cudaSuccess) {
            ytk::set_error("H2D copy of pages failed");
            return YTK_ERR;
        }
        src = reinterpret_cast<const uint8_t*>(h->stage);
    }
    if (ytk::launch_preprocess(src, n_pages, H0, W0, Hn, Wn, e->input, st)) {
        ytk::set_error("preprocess launch failed");
        return YTK_ERR;
    }
    return finish_forward(h, e, prob_out, out_on_device, st);
}

int ytk_dbnet_forward_f32(ytk_dbnet* h, const float* x, int x_on_device, int n, int H, int W, float* prob_out,
                          int out_on_device, void* cuda_stream) {
    std::lock_guard<std::mutex> lk(h->mu);
    DevGuard dev_guard(h->device);  // host threads start on device 0: the handle's device is the one that counts
    cudaStream_t st = static_cast<cudaStream_t>(cuda_stream);
    ytk::DbnetEngine* e = get_engine(h, n, H, W);
    if (!e) return YTK_ERR;
    order_after_previous(h, st);
    const float* src = x;
    if (!x_on_device) {
        const size_t bytes = (size_t)n * 3 * H * W * 4;
        if (ensure_stage(h, bytes)) return YTK_ERR;
        if (cudaMemcpyAsync(h->stage, x, bytes, cudaMemcpyHostToDevice, st) != cudaSuccess) {
            ytk::set_error("H2D copy of input tensor failed");
            return YTK_ERR;
        }
        src = reinterpret_cast<const float*>(h->stage);
    }
    if (ytk::launch_pack_nchw_f32(src, n, H, W, e->input, st)) {
        ytk::set_error("input pack launch failed");
        return YTK_ERR;
    }
    return finish_forward(h, e, prob_out, out_on_device, st);
}

double ytk_dbnet_flops(ytk_dbnet* h, int n_pages, int Hn, int Wn) {
    std::lock_guard<std::mutex> lk(h->mu);
    DevGuard dev_guard(h->device);  // host threads start on device 0: the handle's device is the one that counts
    ytk::DbnetEngine* e = get_engine(h, n_pages, Hn, Wn);
    return e ? e->flops : -1.0;
}

int ytk_dbnet_debug_tensor(ytk_dbnet* h, int n_pages, int Hn, int Wn, const char* name, float* host_out,
                           long long capacity, int* shape4) {
    std::lock_guard<std::mutex> lk(h->mu);
    DevGuard dev_guard(h->device);  // host threads start on device 0: the handle's device is the one that counts
    ytk::DbnetEngine* e = get_engine(h, n_pages, Hn, Wn);
    if (!e) return YTK_ERR;
    auto it = e->dbg.find(name);
    if (it == e->dbg.end() || !it->second.p) {
        ytk::set_error("no debug tensor named '%s'", name);
        return YTK_ERR;
    }
    const ytk::DebugTensor& t = it->second;
    const long long n = (long long)t.n * t.h * t.w * t.c;
    shape4[0] = t.n; shape4[1] = t.h; shape4[2] = t.w; shape4[3] = t.c;
    if (n > capacity) {
        ytk::set_error("debug tensor '%s' needs %lld floats, capacity %lld", name, n, capacity);
        return YTK_ERR;
    }
    cudaDeviceSynchronize();
    if (t.f32) {
        if (cudaMemcpy(host_out, t.p, n * 4, cudaMemcpyDeviceToHost) != cudaSuccess) return YTK_ERR;
    } else {
        float* tmp = nullptr;
        if (cudaMalloc(&tmp, n * 4) != cudaSuccess) return YTK_ERR;
        ytk::launch_op_to_f32(t.p, tmp, n, 0);
        cudaError_t err = cudaMemcpy(host_out, tmp, n * 4, cudaMemcpyDeviceToHost);
        cudaFree(tmp);
        if (err != cudaSuccess) return YTK_ERR;
    }
    return YTK_OK;
}

static_assert(sizeof(ytk_crop_geom) == sizeof(ytk::CropGeom), "ytk_crop_geom and ytk::CropGeom must have one layout");

int ytk_extract_crops_u8(const uint8_t* pages_dev, int n_pages, int H0, int W0, const ytk_crop_geom* geoms, int n_crops,
                         uint8_t* scratch_dev, long long scratch_bytes, uint8_t* canvases_dev, long long canvases_bytes,
                         void* cuda_stream) {
    if (n_crops == 0) return YTK_OK;
    if (!pages_dev || !geoms || !scratch_dev || !canvases_dev || n_pages <= 0 || H0 <= 0 || W0 <= 0 || n_crops < 0) {
        ytk::set_error("ytk_extract_crops_u8: null or empty argument");
        return YTK_ERR;
    }
    long long roi_end = 0;
    for (int i = 0; i < n_crops; ++i) {
        const ytk_crop_geom& g = geoms[i];
        const long long sw = (g.rot & 1) ? g.h : g.w, sh = (g.rot & 1) ? g.w : g.h;
        const bool ok = g.page >= 0 && g.page < n_pages && g.x0 >= 0 && g.y0 >= 0 && g.rw >= 1 && g.rh >= 1 &&
                        (long long)g.x0 + g.rw <= W0 && (long long)g.y0 + g.rh <= H0 && g.w >= 1 && g.h >= 1 &&
                        g.rot >= 0 && g.rot <= 3 && g.cw >= 1 && g.ch >= 1 && g.cw <= sw && g.ch <= sh &&
                        g.cw <= g.canvas_w && g.ch <= g.canvas_h && g.roi_off >= 0 &&
                        g.roi_off + (long long)g.w * g.h * 3 <= scratch_bytes && g.pix_off >= 0 &&
                        g.pix_off + (long long)g.canvas_w * g.canvas_h * 3 <= canvases_bytes;
        if (!ok) {
            ytk::set_error("ytk_extract_crops_u8: inconsistent crop record %d (page %d, roi %d,%d %dx%d, out %dx%d rot %d, "
                           "content %dx%d, canvas %dx%d)", i, g.page, g.x0, g.y0, g.rw, g.rh, g.w, g.h, g.rot, g.cw,
                           g.ch, g.canvas_w, g.canvas_h);
            return YTK_ERR;
        }
        roi_end = std::max(roi_end, g.roi_off + (long long)g.w * g.h * 3);
    }
    // the records are staged in the caller's scratch buffer, 16-byte aligned after the ROIs: no allocation here
    const long long rec_off = (roi_end + 15) / 16 * 16;
    const long long rec_bytes = (long long)n_crops * (long long)sizeof(ytk::CropGeom);
    if (rec_off + rec_bytes > scratch_bytes) {
        ytk::set_error("ytk_extract_crops_u8: scratch_dev holds %lld bytes, need %lld (ROIs) + %lld (records)", scratch_bytes,
                       rec_off, rec_bytes);
        return YTK_ERR;
    }
    cudaPointerAttributes attr;
    if (cudaPointerGetAttributes(&attr, pages_dev) != cudaSuccess || attr.type != cudaMemoryTypeDevice) {
        cudaGetLastError();
        ytk::set_error("ytk_extract_crops_u8: pages_dev is not a device pointer");
        return YTK_ERR;
    }
    DevGuard dev_guard(attr.device);  // host threads start on device 0: the device that owns the pages is the one that counts
    cudaStream_t st = static_cast<cudaStream_t>(cuda_stream);
    ytk::CropGeom* dev = reinterpret_cast<ytk::CropGeom*>(scratch_dev + rec_off);
    cudaError_t err = cudaMemcpyAsync(dev, geoms, (size_t)rec_bytes, cudaMemcpyHostToDevice, st);
    if (err != cudaSuccess) {
        ytk::set_error("ytk_extract_crops_u8: record upload failed: %s", cudaGetErrorString(err));
        return YTK_ERR;
    }
    if (ytk::launch_extract_crops(pages_dev, H0, W0, dev, n_crops, scratch_dev, canvases_dev, st)) {
        ytk::set_error("ytk_extract_crops_u8: kernel launch failed");
        return YTK_ERR;
    }
    return YTK_OK;
}

int ytk_halve_pages_u8(const uint8_t* src_dev, int n_pages, int H, int W, uint8_t* dst_dev, int dH, int dW,
                       void* cuda_stream) {
    // cv2.resize(..., fx=0.5, fy=0.5): dsize = (cvRound(W * 0.5), cvRound(H * 0.5)), round half to even
    const int eh = (int)nearbyint(H * 0.5), ew = (int)nearbyint(W * 0.5);
    if (!src_dev || !dst_dev || n_pages <= 0 || H <= 0 || W <= 0 || dH != eh || dW != ew || dH < 1 || dW < 1) {
        ytk::set_error("ytk_halve_pages_u8: bad arguments (%d pages %dx%d -> %dx%d, expected %dx%d)", n_pages, H, W, dH, dW,
                       eh, ew);
        return YTK_ERR;
    }
    cudaPointerAttributes attr;
    if (cudaPointerGetAttributes(&attr, src_dev) != cudaSuccess || attr.type != cudaMemoryTypeDevice) {
        cudaGetLastError();
        ytk::set_error("ytk_halve_pages_u8: src_dev is not a device pointer");
        return YTK_ERR;
    }
    DevGuard dev_guard(attr.device);
    if (ytk::launch_halve_pages(src_dev, n_pages, H, W, dst_dev, dH, dW, static_cast<cudaStream_t>(cuda_stream))) {
        ytk::set_error("ytk_halve_pages_u8: kernel launch failed");
        return YTK_ERR;
    }
    return YTK_OK;
}

int ytk_parseq_create(const ytk_tensor* tensors, int n_tensors, const ytk_parseq_cfg* cfg, ytk_parseq** out) {
    if (!tensors || !cfg || !out) {
        ytk::set_error("ytk_parseq_create: null argument");
        return YTK_ERR;
    }
    ytk::WeightSet ws;
    for (int i = 0; i < n_tensors; ++i) {
        ytk::TensorView v;
        v.data = tensors[i].data;
        v.ndim = tensors[i].ndim;
        for (int d = 0; d < 4; ++d) v.shape[d] = d < v.ndim ? tensors[i].shape[d] : 1;
        ws.map[tensors[i].name] = v;
    }
    ytk::ParseqCfg c{cfg->embed_dim, cfg->enc_heads, cfg->enc_depth, cfg->patch_h, cfg->patch_w, cfg->img_h,
                     cfg->img_w, cfg->num_tokens, cfg->max_label_length, cfg->dec_heads, cfg->mlp_ratio,
                     cfg->dec_mlp_ratio, cfg->refine_iters, cfg->repetition_stop, cfg->rep_period_max,
                     cfg->rep_min_run_p1, cfg->rep_min_repeats, cfg->decode_ar};
    auto h = std::make_unique<ytk_parseq>();
    cudaGetDevice(&h->device);
    if (h->model.load(ws, c)) return YTK_ERR;
    h->engine.m = &h->model;
    *out = h.release();
    return YTK_OK;
}

void ytk_parseq_destroy(ytk_parseq* h) { delete h; }

void ytk_parseq_set_refine_iters(ytk_parseq* h, int refine_iters) {
    std::lock_guard<std::mutex> lk(h->mu);
    DevGuard dev_guard(h->device);  // host threads start on device 0: the handle's device is the one that counts
    h->model.cfg.refine_iters = refine_iters;
}

int ytk_parseq_forward_crops(ytk_parseq* h, const uint8_t* crops_ptr, int crops_on_device, long long crops_bytes,
                             const ytk_crop* crops, int n_crops, int n_groups, int32_t* ids_out, float* probs_out,
                             int32_t* group_len_out, void* cuda_stream) {
    std::lock_guard<std::mutex> lk(h->mu);
    DevGuard dev_guard(h->device);  // host threads start on device 0: the handle's device is the one that counts
    ytk::ParseqBatch b;
    b.crops = crops_ptr;
    b.crops_on_device = crops_on_device;
    b.crops_bytes = crops_bytes;
    b.ngroups = n_groups;
    b.descs.resize(n_crops);
    const int gh = h->model.gh, pw = h->model.cfg.pw;
    for (int i = 0; i < n_crops; ++i) {
        const ytk_crop& c = crops[i];
        if (c.wp % pw != 0 || c.wp < c.w || c.ntok != gh * (c.wp / pw) || c.group < 0 || c.group >= n_groups ||
            c.wp > h->model.cfg.img_w) {
            ytk::set_error("ytk_parseq_forward_crops: inconsistent crop descriptor %d (w=%d wp=%d ntok=%d group=%d)", i,
                           c.w, c.wp, c.ntok, c.group);
            return YTK_ERR;
        }
        b.descs[i] = ytk::CropDesc{c.pix_off, c.w, c.wp, c.tok_off, c.ntok, c.group};
    }
    return h->engine.forward(b, ids_out, probs_out, group_len_out, nullptr, 0, nullptr,
                             static_cast<cudaStream_t>(cuda_stream))
               ? YTK_ERR
               : YTK_OK;
}

int ytk_parseq_forward_f32(ytk_parseq* h, const float* images, int images_on_device, int B, int W, float* logits_out,
                           int logits_on_device, int32_t* ids_out, float* probs_out, int32_t* steps_out,
                           int32_t* rep_cut_out, float* memory_out, void* cuda_stream) {
    std::lock_guard<std::mutex> lk(h->mu);
    DevGuard dev_guard(h->device);  // host threads start on device 0: the handle's device is the one that counts
    const int pw = h->model.cfg.pw, gh = h->model.gh;
    if (W % pw != 0 || W > h->model.cfg.img_w || W <= 0) {
        ytk::set_error("ytk_parseq_forward_f32: width %d must be a positive multiple of %d and <= %d", W, pw,
                       h->model.cfg.img_w);
        return YTK_ERR;
    }
    ytk::ParseqBatch b;
    b.images_f32 = images;
    b.images_on_device = images_on_device;
    b.image_w = W;
    b.crops_bytes = images_on_device ? 0 : (long long)B * 3 * 32 * W * 4;
    b.ngroups = 1;
    b.descs.resize(B);
    const int ntok = gh * (W / pw);
    for (int i = 0; i < B; ++i) b.descs[i] = ytk::CropDesc{0, W, W, i * ntok, ntok, 0};
    int glen = 0;
    cudaStream_t st = static_cast<cudaStream_t>(cuda_stream);
    if (h->engine.forward(b, ids_out, probs_out, &glen, logits_out, logits_on_device, memory_out, st)) return YTK_ERR;
    if (steps_out) *steps_out = glen;
    if (rep_cut_out) {
        if (cudaMemcpy(rep_cut_out, h->engine.ar.rep_cut, sizeof(int) * B, cudaMemcpyDeviceToHost) != cudaSuccess) {
            ytk::set_error("rep_cut copy failed");
            return YTK_ERR;
        }
    }
    return YTK_OK;
}

double ytk_parseq_last_flops(ytk_parseq* h) { return h->engine.flops; }
int ytk_parseq_last_steps(ytk_parseq* h) { return h->engine.last_steps; }
void ytk_parseq_last_phase_ms(ytk_parseq* h, float* ms4) {
    for (int i = 0; i < 4; ++i) ms4[i] = h->engine.phase_ms[i];
}

}  // extern "C"


// ------------------------------------------------------------------------------------------------ RT-DETRv2
struct ytk_rtdetr {
    ytk::RtdetrModel model;
    std::map<int, std::unique_ptr<ytk::RtdetrEngine>> engines;   // per batch size
    std::mutex mu;
    int device = 0;
    cudaEvent_t last_done = nullptr;   // buffers of an engine are shared by all calls: order them (see ytk_dbnet)
};

static ytk::RtdetrEngine* rt_engine(ytk_rtdetr* h, int n) {
    auto it = h->engines.find(n);
    if (it != h->engines.end()) return it->second.get();
    if (h->engines.size() >= 4) {
        cudaDeviceSynchronize();
        h->engines.erase(h->engines.begin());
    }
    auto e = std::make_unique<ytk::RtdetrEngine>();
    if (e->build(h->model, n)) return nullptr;
    ytk::RtdetrEngine* p = e.get();
    h->engines[n] = std::move(e);
    return p;
}

int ytk_rtdetr_create(const ytk_tensor* tensors, int n_tensors, int num_classes, int num_queries, int img_size,
                      ytk_rtdetr** out) {
    if (!tensors || !out) {
        ytk::set_error("ytk_rtdetr_create: null argument");
        return YTK_ERR;
    }
    ytk::WeightSet ws;
    for (int i = 0; i < n_tensors; ++i) {
        ytk::TensorView v;
        v.data = tensors[i].data;
        v.ndim = tensors[i].ndim;
        for (int d = 0; d < 4; ++d) v.shape[d] = d < v.ndim ? tensors[i].shape[d] : 1;
        ws.map[tensors[i].name] = v;
    }
    auto h = std::make_unique<ytk_rtdetr>();
    cudaGetDevice(&h->device);
    ytk::RtCfg cfg;
    cfg.num_classes = num_classes;
    cfg.num_queries = num_queries;
    cfg.img = img_size;
    if (num_classes < 1 || num_classes > 8 || num_queries < 1) {
        ytk::set_error("ytk_rtdetr_create: num_classes %d (1..8) / num_queries %d unsupported", num_classes, num_queries);
        return YTK_ERR;
    }
    if (h->model.load(ws, cfg)) return YTK_ERR;
    *out = h.release();
    return YTK_OK;
}

void ytk_rtdetr_destroy(ytk_rtdetr* h) {
    if (!h) return;
    DevGuard dev_guard(h->device);
    if (h->last_done) {
        cudaEventSynchronize(h->last_done);
        cudaEventDestroy(h->last_done);
    }
    cudaDeviceSynchronize();
    delete h;
}

int ytk_rtdetr_device(const ytk_rtdetr* h) { return h ? h->device : -1; }

int ytk_rtdetr_forward_f32(ytk_rtdetr* h, const float* x, int x_on_device, int n, float* pred_logits, float* pred_boxes,
                           int out_on_device, void* cuda_stream) {
    if (!h || !x || !pred_logits || !pred_boxes || n < 1) {
        ytk::set_error("ytk_rtdetr_forward_f32: null or empty argument");
        return YTK_ERR;
    }
    std::lock_guard<std::mutex> lk(h->mu);
    DevGuard dev_guard(h->device);
    cudaStream_t st = static_cast<cudaStream_t>(cuda_stream);
    ytk::RtdetrEngine* e = rt_engine(h, n);
    if (!e) return YTK_ERR;
    if (h->last_done) cudaStreamWaitEvent(st, h->last_done, 0);
    const int S = h->model.cfg.img, K = h->model.cfg.num_queries, C = h->model.cfg.num_classes;
    const float* src = x;
    if (!x_on_device) {
        if (cudaMemcpyAsync(e->in_f32, x, (size_t)n * 3 * S * S * 4, cudaMemcpyHostToDevice, st) != cudaSuccess) {
            ytk::set_error("H2D copy of the input tensor failed");
            return YTK_ERR;
        }
        src = e->in_f32;
    }
    if (ytk::launch_rt_pack_input(src, n, S, S, e->input, st) || e->run(st)) return YTK_ERR;
    const cudaMemcpyKind kind = out_on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost;
    cudaError_t err = cudaMemcpyAsync(pred_logits, e->out_logits, (size_t)n * K * C * 4, kind, st);
    if (err == cudaSuccess) err = cudaMemcpyAsync(pred_boxes, e->boxes, (size_t)n * K * 16, kind, st);
    if (!h->last_done) cudaEventCreateWithFlags(&h->last_done, cudaEventDisableTiming);
    if (h->last_done) cudaEventRecord(h->last_done, st);
    if (err == cudaSuccess && !out_on_device) err = cudaStreamSynchronize(st);
    if (err != cudaSuccess) {
        ytk::set_error("RT-DETRv2 output copy failed: %s", cudaGetErrorString(err));
        return YTK_ERR;
    }
    return YTK_OK;
}

double ytk_rtdetr_flops(ytk_rtdetr* h, int n) {
    std::lock_guard<std::mutex> lk(h->mu);
    DevGuard dev_guard(h->device);
    ytk::RtdetrEngine* e = rt_engine(h, n);
    return e ? e->flops : -1.0;
}

long long ytk_rtdetr_device_bytes(ytk_rtdetr* h, int n) {
    std::lock_guard<std::mutex> lk(h->mu);
    DevGuard dev_guard(h->device);
    ytk::RtdetrEngine* e = rt_engine(h, n);
    return e ? (long long)e->total_bytes : -1;
}

int ytk_rtdetr_debug_tensor(ytk_rtdetr* h, int n, const char* name, float* host_out, long long capacity, int* shape4) {
    std::lock_guard<std::mutex> lk(h->mu);
    DevGuard dev_guard(h->device);
    ytk::RtdetrEngine* e = rt_engine(h, n);
    if (!e) return YTK_ERR;
    auto it = e->dbg.find(name);
    if (it == e->dbg.end() || !it->second.p) {
        ytk::set_error("no debug tensor named '%s'", name);
        return YTK_ERR;
    }
    const ytk::DebugTensor& t = it->second;
    const long long cnt = (long long)t.n * t.h * t.w * t.c;
    shape4[0] = t.n; shape4[1] = t.h; shape4[2] = t.w; shape4[3] = t.c;
    if (cnt > capacity) {
        ytk::set_error("debug tensor '%s' needs %lld floats, capacity %lld", name, cnt, capacity);
        return YTK_ERR;
    }
    cudaDeviceSynchronize();
    if (t.f32) {
        if (cudaMemcpy(host_out, t.p, cnt * 4, cudaMemcpyDeviceToHost) != cudaSuccess) return YTK_ERR;
    } else {
        float* tmp = nullptr;
        if (cudaMalloc(&tmp, cnt * 4) != cudaSuccess) return YTK_ERR;
        ytk::launch_op_to_f32(t.p, tmp, cnt, 0);
        cudaError_t err = cudaMemcpy(host_out, tmp, cnt * 4, cudaMemcpyDeviceToHost);
        cudaFree(tmp);
        if (err != cudaSuccess) return YTK_ERR;
    }
    return YTK_OK;
}
