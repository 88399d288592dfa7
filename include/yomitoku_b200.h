/*
 * yomitoku_b200 C ABI (libytk_b200.so) - the drop-in boundary for the DBNet -> PARSeq hot path.
 *
 * The reference (kotaro-kinoshita/yomitoku) has no FFI: its seam is the Python object protocol
 * `self.model(tensor)` inside TextDetector / TextRecognizer (reference src/yomitoku/text_detector.py:127-131,
 * src/yomitoku/text_recognizer.py:247-256, SURVEY.md section 8b).  These entry points are what a ctypes binding
 * behind those two call sites binds to; INTEGRATION.md shows the stub.  Plain pointers and sizes only, no torch
 * types; all device pointers are caller-owned; every call returns 0 on success and a nonzero code on failure, with a
 * human-readable message from ytk_last_error() (thread-local).  No exceptions cross this boundary.
 */
#ifndef YOMITOKU_B200_H
#define YOMITOKU_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define YTK_OK 0
#define YTK_ERR 1

/* activation codes for the op-level entry points */
#define YTK_ACT_NONE 0
#define YTK_ACT_RELU 1
#define YTK_ACT_GELU 2
#define YTK_ACT_SIGMOID 3
#define YTK_ACT_SILU 4

const char* ytk_last_error(void);
int ytk_version(void);
/* number of kernel launches issued by this library on the calling process since load (bench.py gpu_launches) */
long long ytk_launch_count(void);
/* Measurement aid (bench.py roofline): between begin and end every gemm_tc_kernel launch is bracketed by CUDA events on
 * its own stream; end returns the summed algorithmic FLOPs, summed kernel durations (ms) and the launch count. */
void ytk_gemm_profile_begin(void);
int ytk_gemm_profile_end(double* flops, double* ms, long long* launches);

/* ---- op level (kernel parity tests; replaces the cuDNN/cuBLAS call sites listed in SURVEY.md section 2.3) ----
 * Convolution as tcgen05 implicit GEMM.  in: NHWC fp16 [N,H,W,in_ld] (first Cin channels used), w: fp16
 * [Cout][kh][kw][Cin], bias fp32 [Cout] or NULL, resid: [N,Ho,Wo,ldr] fp16/fp32 or NULL, out: [N,Ho,Wo,ldc]
 * fp16/fp32.  Replaces torch.nn.Conv2d + BatchNorm2d(eval, folded) + ReLU (+ residual add) of
 * torchvision ResNet-50 bottlenecks (reference models/dbnet_plus.py:30-38) and the decoder convs (:56-116).
 * mode 1 = ConvTranspose2d(kernel 2, stride 2) written as a GEMM with a pixel-shuffle epilogue (:111,:114). */
int ytk_op_conv2d_f16(const void* in, int N, int H, int W, int Cin, long long in_ld, const void* w, const float* bias,
                       int kh, int kw, int stride, int pad, int dil, int Cout, const void* resid, int resid_f32,
                       long long ldr, void* out, int out_f32, long long ldc, int act, int mode, void* cuda_stream);

/* Linear layer y = act(A W^T + b (+ resid)); A [M,lda] fp16, W [N,K] fp16 (torch nn.Linear layout), K % 64 == 0.
 * Replaces nn.Linear / timm Mlp / attention projections (reference models/layers/parseq_transformer.py:43-52,
 * models/parseq.py:72). */
int ytk_op_linear_f16(const void* A, long long lda, int M, int K, const void* W, int N, const float* bias,
                       const void* resid, int resid_f32, long long ldr, void* out, int out_f32, long long ldc, int act,
                       void* cuda_stream);

/* One descriptor per packed sequence of ytk_op_attention_f16 (the layout of ytk::SeqDesc, csrc/parseq_ops.h). */
typedef struct ytk_attn_seq {
    int32_t q_off;     /* first query row in Q */
    int32_t q_len;
    int32_t o_off;     /* first output row in O */
    int32_t k_len;     /* number of keys */
    long long k_base;  /* element offset of key 0 inside K / V (key j at k_base + j * ldkv; a multiple of ldkv) */
    int32_t kpad;      /* masked mode: keys >= kpad are padding */
    int32_t pad_;
} ytk_attn_seq;

/* softmax(Q K^T / sqrt(head_dim)) V per (sequence, head) over packed ragged sequences; Q [q_rows, ldq], K / V
 * [kv_rows, ldkv], O [*, ldo] fp16 on the device, head h = columns [h*head_dim, (h+1)*head_dim); seqs_dev: device array.
 * masked != 0: key j visible to query i iff (i < 2 || j <= i) && j < kpad (PARSeq refinement mask, reference
 * models/parseq.py:267-297).  impl: 0 default (tcgen05 kernel), 1 legacy mma.sync kernel, 2/3 tcgen05 kernel with the
 * V-descriptor convention forced.  Replaces timm Attention's F.scaled_dot_product_attention (reference
 * models/layers/parseq_transformer.py:206-234) and nn.MultiheadAttention's core (parseq_transformer.py:83-92). */
int ytk_op_attention_f16(const void* Q, long long ldq, long long q_rows, const void* K, const void* V, long long ldkv,
                         long long kv_rows, void* O, long long ldo, const ytk_attn_seq* seqs_dev, int nseq, int max_q_len,
                         int heads, int head_dim, int masked, int impl, void* cuda_stream);

/* RT-DETRv2 query selection: per image, the indices of the K largest of L fp32 scores in descending order, equal scores
 * by ascending index (torch.topk(scores, K) of reference models/layers/rtdetrv2_decoder.py:730).  scores_dev
 * [n_img, L] and out_idx_dev [n_img, K] int32 are device memory.  L <= 16384: one bitonic sort in shared memory; up to
 * L = 45056 with K <= 2048: radix select + sort of the K selected (the 960 x 960 cell detector has L = 18900, K = 1500).
 * Other sizes return an error. */
int ytk_op_rt_topk_f32(const float* scores_dev, int n_img, int L, int K, int* out_idx_dev, void* stream);

/* ---- Device-side front half of the DBNet post-processing (reference postprocessor/dbnet_postporcessor.py:39-82:
 * binarize, findContours, and the pixel work of minAreaRect / box_score_fast).  One record per horizontal run of an
 * 8-connected component of (prob > thresh). ---- */
typedef struct ytk_db_run {
    int32_t root;  /* raster index of the component's first pixel: component id; OpenCV lists outer contours in
                      descending order of it */
    int32_t y;
    int32_t x0;    /* first column */
    int32_t x1;    /* last column, inclusive */
    double sum;    /* sum of prob over the run */
} ytk_db_run;

/* prob_dev: [n_pages, H, W] fp32 device; scratch_dev: n_pages*H*W*4 bytes device; runs_dev: [n_pages, max_runs_per_page]
 * device; meta_dev: [n_pages, 4] int32 device = {runs found (> max_runs_per_page means truncated), components,
 * 4 * Euler number (8-connectivity: holes = components - Euler number), overflow flag}.  Asynchronous on the stream.
 * The end points of a component's runs have the same minAreaRect as its OpenCV contour, sum / pixel count of the runs is
 * box_score_fast of a component without holes; pages with holes must use the host path (the caller's decision). */
int ytk_dbnet_post_front(const float* prob_dev, int n_pages, int H, int W, float thresh, void* scratch_dev,
                         long long scratch_bytes, ytk_db_run* runs_dev, int max_runs_per_page, int32_t* meta_dev,
                         void* cuda_stream);

/* ---- DBNet text detector: replaces `self.model(tensor)` in reference TextDetector.__call__
 * (src/yomitoku/text_detector.py:127-129 -> models/dbnet_plus.py:243-246) and, in the fused u8 entry, also
 * TextDetector.preprocess (text_detector.py:99-107, data/functions.py:196-264). ---- */
typedef struct ytk_dbnet ytk_dbnet;

/* One entry of the reference-keyed state_dict (host fp32, SURVEY.md Appendix C; the strict key set of
 * DBNet.state_dict() / PARSeq.state_dict() as stored in the HF model.safetensors). */
typedef struct {
    const char* name;
    const float* data;
    int ndim;
    long long shape[4];
} ytk_tensor;

/* Folds BatchNorm, repacks weights to NHWC fp16 and uploads them.  shortest_size / limit_size are cfg.data.* of the
 * detector config (reference configs/cfg_text_detector_dbnet_v2_1.py:23-26). */
int ytk_dbnet_create(const ytk_tensor* tensors, int n_tensors, int shortest_size, int limit_size, ytk_dbnet** out);
void ytk_dbnet_destroy(ytk_dbnet* h);
/* CUDA device ordinal a handle is bound to (the device that was current at create()). */
int ytk_dbnet_device(const ytk_dbnet* h);
/* network input size for an H0 x W0 page = reference resize_shortest_edge (data/functions.py:212-224) */
int ytk_dbnet_input_size(const ytk_dbnet* h, int H0, int W0, int* Hn, int* Wn);
/* pages: [n_pages, H0, W0, 3] uint8 BGR (caller-owned; device pointer iff pages_on_device, else host - pinned for
 * async copies).  prob_out: [n_pages, Hn, Wn] fp32 sigmoid map = preds["binary"][:, 0] of the reference. */
int ytk_dbnet_forward_u8(ytk_dbnet* h, const uint8_t* pages, int pages_on_device, int n_pages, int H0, int W0,
                         float* prob_out, int out_on_device, void* cuda_stream);
/* model-level seam: x = normalised (n,3,H,W) fp32 exactly as the reference feeds DBNet.forward; H, W % 32 == 0 */
int ytk_dbnet_forward_f32(ytk_dbnet* h, const float* x_nchw, int x_on_device, int n, int H, int W, float* prob_out,
                          int out_on_device, void* cuda_stream);
/* algorithmic conv FLOPs (2*MAC) of one forward at this shape (roofline accounting) */
double ytk_dbnet_flops(ytk_dbnet* h, int n_pages, int Hn, int Wn);
/* test hook: copy a named intermediate activation (NHWC) of the last run at this shape to host fp32.
 * shape4 receives n,h,w,c.  Names: stem, pool, layer1..layer4, layerL.B, f1..f4, fuse, asf_a, bin1, bin2, prob. */
int ytk_dbnet_debug_tensor(ytk_dbnet* h, int n_pages, int Hn, int Wn, const char* name, float* host_out,
                           long long capacity, int* shape4);

/* ---- PARSeq text recognizer: replaces `self.model(data).softmax(-1)` + tokenizer arg-max in reference
 * TextRecognizer._run_inference / postprocess (src/yomitoku/text_recognizer.py:247-256, 232-245 ->
 * models/parseq.py:159-311, postprocessor/parseq_tokenizer.py:64-88). ---- */
typedef struct ytk_parseq ytk_parseq;

/* values of the recognizer config (reference configs/cfg_text_recognizer_parseq*.py) + repetition-stop knobs
 * (models/parseq.py:93-96) */
typedef struct {
    int embed_dim, enc_heads, enc_depth, patch_h, patch_w, img_h, img_w, num_tokens, max_label_length, dec_heads,
        mlp_ratio, dec_mlp_ratio, refine_iters, repetition_stop, rep_period_max, rep_min_run_p1, rep_min_repeats,
        decode_ar; /* cfg.decode_ar (models/parseq.py:192,252): 0 = one non-autoregressive pass instead of the AR loop */
} ytk_parseq_cfg;

/* One crop of a packed recognizer call.  The canvas is the reference's `dataset.data[i]` (RGB uint8, 32 rows,
 * w columns, black padded, data/functions.py:379-439); wp is the width the reference's _collate would pad it to
 * (max width of its mini-batch, text_recognizer.py:146-156); group = index of that mini-batch (the AR loop stops
 * per mini-batch, models/parseq.py:245-250). */
typedef struct {
    long long pix_off; /* byte offset of the canvas in the packed buffer */
    int w;             /* stored canvas width */
    int wp;            /* padded width (multiple of patch_w, >= w) */
    int tok_off;       /* first encoder token row of this crop (crops are packed back to back) */
    int ntok;          /* (32 / patch_h) * (wp / patch_w) */
    int group;
} ytk_crop;

int ytk_parseq_create(const ytk_tensor* tensors, int n_tensors, const ytk_parseq_cfg* cfg, ytk_parseq** out);
void ytk_parseq_destroy(ytk_parseq* h);
int ytk_parseq_device(const ytk_parseq* h);
void ytk_parseq_set_refine_iters(ytk_parseq* h, int refine_iters);
/* crops: packed canvases; host pointer (pinned memory for async copies) or, iff crops_on_device, a device pointer
 * (the copy is skipped).  Outputs (host): ids / probs
 * [n_crops, max_label_length + 1] = per-position arg-max token and its softmax probability (what
 * BaseTokenizer.decode computes from the full distribution), group_len [n_groups] = AR steps each mini-batch ran
 * (= number of valid positions when refine_iters == 0). */
int ytk_parseq_forward_crops(ytk_parseq* h, const uint8_t* crops, int crops_on_device, long long crops_bytes,
                             const ytk_crop* descs, int n_crops, int n_groups, int32_t* ids_out, float* probs_out,
                             int32_t* group_len_out, void* cuda_stream);
/* model-level seam: images (B,3,32,W) fp32 as fed to PARSeq.forward (one mini-batch).  logits_out (optional)
 * receives (B, S, C) fp32, S = max_label_length + 1 (only the first group_len positions are written when
 * refine_iters == 0), WITHOUT the repetition patch; rep_cut_out [B] (-1 = none) lets the caller apply
 * models/parseq.py:301-309.  memory_out (optional, host) receives the encoder output (B*N, D) fp32. */
int ytk_parseq_forward_f32(ytk_parseq* h, const float* images, int images_on_device, int B, int W, float* logits_out,
                           int logits_on_device, int32_t* ids_out, float* probs_out, int32_t* steps_out,
                           int32_t* rep_cut_out, float* memory_out, void* cuda_stream);
/* algorithmic FLOPs (2*MAC; GEMMs + attention) and AR steps of the last forward call */
double ytk_parseq_last_flops(ytk_parseq* h);
int ytk_parseq_last_steps(ytk_parseq* h);
/* CUDA-event times (ms) of the last forward: encoder, AR decode, refinement, output copies */
void ytk_parseq_last_phase_ms(ytk_parseq* h, float* ms4);

/* ---- Device-side crop extraction: replaces the pixel work of ParseqDataset._preprocess_on (reference
 * src/yomitoku/data/dataset.py:106-123): extract_roi_with_perspective (data/functions.py:301-333, cv2.warpPerspective),
 * rotate_text_image (:336-350) and resize_with_padding / resize_with_dynamic_padding (:379-439, cv2.resize INTER_AREA +
 * paste on a black canvas), bit-exact with OpenCV 4.13 for 8UC3.  The scalar decisions (bounding box, output size,
 * rotation, content and canvas size, the inverse perspective matrix) stay on the host: one record per crop
 * (yomitoku_b200/data.py: crop_geometry).  The canvases come out packed exactly as ytk_parseq_forward_crops takes them
 * with crops_on_device = 1, so no crop pixel leaves the GPU. ---- */
typedef struct {
    double minv[9];    /* cv2.invert(cv2.getPerspectiveTransform(quad - (x0,y0), [[0,0],[w,0],[w,h],[0,h]])), row major */
    long long roi_off; /* byte offset of this crop's rectified ROI in scratch_dev: w*h*3 bytes */
    long long pix_off; /* byte offset of this crop's canvas in canvases_dev: canvas_h*canvas_w*3 bytes, RGB */
    int page;          /* index into pages_dev */
    int x0, y0, rw, rh; /* bounding-box slice of the (int64-truncated) quad inside the page */
    int w, h;          /* rectified size: (int |p0p1|, int |p1p2|) */
    int rot;           /* bit 0: rotate 90 degrees counter-clockwise after the warp (h > 2w); bit 1: then rotate by 180
                          degrees (the orientation fallback's second look, text_recognizer.py:319-328) */
    int cw, ch;        /* content size after the down-scale-only fit (calc_resize_without_padding) */
    int canvas_w, canvas_h;
} ytk_crop_geom;

/* pages_dev: [n_pages, H0, W0, 3] uint8 BGR in device memory (e.g. the buffer handed to ytk_dbnet_forward_u8 with
 * pages_on_device = 1); geoms: host array (pageable: may be reused as soon as the call returns; page-locked: must stay
 * valid until the stream has passed the call); scratch_dev / canvases_dev: caller-owned device buffers.  scratch_dev
 * holds the rectified ROIs (at roi_off) and, 16-byte aligned after the last ROI, a copy of the n_crops records, so
 * scratch_bytes >= align16(max(roi_off + w*h*3)) + n_crops * sizeof(ytk_crop_geom): the call allocates nothing.
 * Asynchronous on cuda_stream: one H2D copy of the records + two kernel launches. */
int ytk_extract_crops_u8(const uint8_t* pages_dev, int n_pages, int H0, int W0, const ytk_crop_geom* geoms, int n_crops,
                         uint8_t* scratch_dev, long long scratch_bytes, uint8_t* canvases_dev, long long canvases_bytes,
                         void* cuda_stream);

/* One level of the recognizer's source_downscale pyramid (reference data/dataset.py:64-86):
 * cv2.resize(page, None, fx=0.5, fy=0.5, interpolation=cv2.INTER_AREA) for n_pages pages [n, H, W, 3] uint8 in device
 * memory, bit-exact with OpenCV 4.13 (2x2 cells round half up; the clipped last column / row of an odd size averages
 * the pixels that exist).  dH = cvRound(H / 2), dW = cvRound(W / 2) (round half to even) - anything else is rejected. */
int ytk_halve_pages_u8(const uint8_t* src_dev, int n_pages, int H, int W, uint8_t* dst_dev, int dH, int dW,
                       void* cuda_stream);

/* ---- RT-DETRv2 layout parser / table structure recognizer: replaces `self.model(img_tensor)` in reference
 * LayoutParser.__call__ (src/yomitoku/layout_parser.py:258-262 -> models/rtdetr.py:17-22) and
 * TableStructureRecognizer.__call__ (table_structure_recognizer.py:272-276).  One architecture, two weight sets
 * (num_classes 6 / 3). ---- */
typedef struct ytk_rtdetr ytk_rtdetr;

/* tensors: the reference's state_dict (RTDETRv2(cfg).state_dict() keys, host fp32; the boolean `decoder.valid_mask` may
 * be passed as 0/1 floats or left out - it is derived from the finite entries of `decoder.anchors`).  img_size: the square
 * evaluation size (cfg.data.img_size = eval_spatial_size, 640). */
int ytk_rtdetr_create(const ytk_tensor* tensors, int n_tensors, int num_classes, int num_queries, int img_size,
                      ytk_rtdetr** out);
void ytk_rtdetr_destroy(ytk_rtdetr* h);
int ytk_rtdetr_device(const ytk_rtdetr* h);
/* x: [n, 3, img, img] fp32 in [0, 1] (what the reference's transforms produce), host or device.
 * pred_logits: [n, num_queries, num_classes] fp32, pred_boxes: [n, num_queries, 4] fp32 (cx, cy, w, h in [0, 1]) - the
 * "pred_logits" / "pred_boxes" of the reference's output dict, rows in the decoder's query order (descending encoder
 * score).  Outputs on the host: the call returns after the copy; on the device: asynchronous on the stream. */
int ytk_rtdetr_forward_f32(ytk_rtdetr* h, const float* x, int x_on_device, int n, float* pred_logits, float* pred_boxes,
                           int out_on_device, void* cuda_stream);
double ytk_rtdetr_flops(ytk_rtdetr* h, int n);
/* device bytes of the activation buffers of the batch-n launch plan (built on first use, like a forward), -1 on error */
long long ytk_rtdetr_device_bytes(ytk_rtdetr* h, int n);
/* test hook: copies an intermediate activation (by name, see rtdetr_engine.cu) of the LAST forward of batch size n to
 * the host as fp32; shape4 = {n, h, w, c} (token matrices: {1, 1, rows, c}) */
int ytk_rtdetr_debug_tensor(ytk_rtdetr* h, int n, const char* name, float* host_out, long long capacity, int* shape4);

#ifdef __cplusplus
}
#endif
#endif /* YOMITOKU_B200_H */
