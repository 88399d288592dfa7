// Launchers of the non-GEMM RT-DETRv2 kernels (rtdetr_ops.cu).  All return 0 on success.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace ytk {

// The decoder's multi-scale memory.  Token matrices are LEVEL-MAJOR: rows [off[l] * n_img, off[l + 1] * n_img) hold
// level l of every image (image-major inside the level, raster order inside the image) - each level is exactly the NHWC
// output of its 1x1 input projection, so no flatten / concat copy exists.  An "anchor" is the reference's token index
// inside one image: off[l] + y * w[l] + x (rtdetrv2_decoder.py:620-637).
struct RtLevels {
    static constexpr int kMax = 4;
    int n = 0;
    int h[kMax], w[kMax], off[kMax + 1], points[kMax];
    int total = 0;       // anchors per image
};

__host__ __device__ inline long long rt_anchor_row(const RtLevels& lv, int n_img, int img, int anchor) {
    int l = 0;
    while (l + 1 < lv.n && anchor >= lv.off[l + 1]) ++l;
    return (long long)lv.off[l] * n_img + (long long)img * lv.h[l] * lv.w[l] + (anchor - lv.off[l]);
}
__host__ __device__ inline int rt_row_anchor_img(const RtLevels& lv, int n_img, long long row, int* img) {
    int l = 0;
    while (l + 1 < lv.n && row >= (long long)lv.off[l + 1] * n_img) ++l;
    const long long r = row - (long long)lv.off[l] * n_img;
    const int hw = lv.h[l] * lv.w[l];
    *img = (int)(r / hw);
    return lv.off[l] + (int)(r % hw);
}
__host__ __device__ inline int rt_row_anchor(const RtLevels& lv, int n_img, long long row) {
    int img;
    return rt_row_anchor_img(lv, n_img, row, &img);
}

int launch_rt_pack_input(const float* src_nchw, int n_img, int H, int W, void* dst_nhwc64, cudaStream_t st);
int launch_rt_avgpool2(const void* in, void* out, int n_img, int H, int W, int C, cudaStream_t st);
// nearest x2 of src [n, Hs, Ws, C] (row pitch lds elements) into channels [coff, coff + C) of dst [n, 2Hs, 2Ws, ldd]
int launch_rt_upsample_nearest2(const void* src, long long lds, int n_img, int Hs, int Ws, int C, void* dst, long long ldd,
                                int coff, cudaStream_t st);
// out = a + b (fp16 [rows, C]); with b_f32: out = a + b_f32[row % period] (fp32 table [period, C])
int launch_rt_add(const void* a, const void* b, const float* b_f32, int C, int period, void* out, long long rows,
                  cudaStream_t st);
// x[row(anchor, img), :] = bias for the anchors listed in `invalid` (device array of anchor ids)
int launch_rt_mask_invalid(float* x, int D, const float* bias, const int* invalid, int n_invalid, const RtLevels& lv,
                           int n_img, cudaStream_t st);
int launch_rt_enc_scores(const float* logits, long long ldl, int C, const RtLevels& lv, int n_img, float* scores,
                         cudaStream_t st);
// per image: indices of the K largest of L scores, descending (ties: smaller index first).  A bitonic sort of all L keys
// in shared memory when next_pow2(L) 8-byte keys fit kTopkSmemBytes (L <= 16384: the 640 models), otherwise
// launch_rt_topk_select.
constexpr int kTopkSmemBytes = 200 * 1024;
int launch_rt_topk(const float* scores, int n_img, int L, int K, int* out_idx, cudaStream_t st);
// The same result by radix select + a sort of the K selected keys: needs 1 <= K <= min(L, kTopkSelectMaxK) and
// L <= kTopkSelectMaxL (4 B per score + 8 B per next_pow2(K) key + 1 KB of histogram within kTopkSmemBytes; the kernel's
// key keeps 16 anchor bits).  Other sizes return an error.
constexpr int kTopkSelectMaxK = 2048;
constexpr int kTopkSelectMaxL = 45056;
static_assert(kTopkSelectMaxL <= 65536, "topk_select_kernel keeps 16 anchor bits");
static_assert(kTopkSelectMaxL * 4 + kTopkSelectMaxK * 8 + 1024 <= kTopkSmemBytes, "topk_select_kernel shared memory");
int launch_rt_topk_select(const float* scores, int n_img, int L, int K, int* out_idx, cudaStream_t st);
int launch_rt_gather_queries(const float* om, int D, const int* idx, int K, const RtLevels& lv, int n_img, float* tgt,
                             void* tgt16, const float* anchors, float* anchor_sel, cudaStream_t st);
// ref[i] = sigmoid(delta[i] + (anchor_sel ? anchor_sel[i] : inverse_sigmoid(ref[i]))), i over n boxes x 4
int launch_rt_ref_update(const float* delta, long long ldd, const float* anchor_sel, float* ref, int n, cudaStream_t st);
int launch_rt_qpos_l0(const float* ref, const float* W, const float* b, int H1, void* out, int rows, cudaStream_t st);
int launch_rt_deform_attn(const float* ow, long long ldo, const float* ref, const void* value, long long ldv, int voff,
                          const RtLevels& lv, int n_img, int K, int heads, int head_dim, float offset_scale, void* out,
                          long long ldout, cudaStream_t st);
int launch_rt_copy_cols(const float* src, long long ld, int C, float* dst, long long rows, cudaStream_t st);

}  // namespace ytk
