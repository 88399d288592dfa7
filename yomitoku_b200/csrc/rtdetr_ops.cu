// Non-GEMM kernels of the RT-DETRv2 engine (rtdetr_engine.cu): input packing, average pooling of the variant-d shortcuts,
// nearest up-sampling into the FPN concat buffers, element-wise adds, query selection (top-k), reference-box updates and
// the multi-scale deformable attention sampling.  Replaces the torch ops of reference
// models/layers/rtdetr_backbone.py:118-131, rtdetr_hybrid_encoder.py:380-393, rtdetrv2_decoder.py:36-40, 155-222,
// 306-388, 680-746.  HBM / latency bound byte work; every activation is NHWC fp16, the decoder state is fp32.
#include "rtdetr_ops.h"

#include <cmath>

#include "gemm_tc.h"
#include "ptx.cuh"

namespace ytk {

namespace {

__device__ __forceinline__ void unpack8(const uint4& u, float* f) {
    f[0] = op_lo(u.x); f[1] = op_hi(u.x); f[2] = op_lo(u.y); f[3] = op_hi(u.y);
    f[4] = op_lo(u.z); f[5] = op_hi(u.z); f[6] = op_lo(u.w); f[7] = op_hi(u.w);
}
__device__ __forceinline__ uint4 pack8(const float* f) {
    uint4 u;
    u.x = pack_op(f[0], f[1]); u.y = pack_op(f[2], f[3]); u.z = pack_op(f[4], f[5]); u.w = pack_op(f[6], f[7]);
    return u;
}

// (n,3,H,W) fp32 in [0,1] (what the reference's ToTensor produces) -> NHWC with 64 channels (3 real), one thread per
// (pixel, 8-channel group)
__global__ void pack_input_kernel(const float* __restrict__ src, int n_img, int H, int W, uint4* __restrict__ dst) {
    const long long total = (long long)n_img * H * W * 8;
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= total) return;
    const int g = (int)(idx & 7);
    const long long pix = idx >> 3;
    float o[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    if (g == 0) {
        const int w = (int)(pix % W), h = (int)((pix / W) % H), img = (int)(pix / ((long long)W * H));
#pragma unroll
        for (int c = 0; c < 3; ++c) o[c] = __ldg(src + (((size_t)img * 3 + c) * H + h) * W + w);
    }
    dst[idx] = pack8(o);
}

// AvgPool2d(2, 2, ceil_mode) for even sizes: NHWC fp16, one thread per (output pixel, 8-channel group)
__global__ void avgpool2_kernel(const uint4* __restrict__ in, uint4* __restrict__ out, int n_img, int H, int W, int C8) {
    const int Ho = H / 2, Wo = W / 2;
    const long long total = (long long)n_img * Ho * Wo * C8;
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= total) return;
    const int c = (int)(idx % C8);
    const int wo = (int)((idx / C8) % Wo);
    const int ho = (int)((idx / ((long long)C8 * Wo)) % Ho);
    const int img = (int)(idx / ((long long)C8 * Wo * Ho));
    float acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
#pragma unroll
    for (int dy = 0; dy < 2; ++dy)
#pragma unroll
        for (int dx = 0; dx < 2; ++dx) {
            float f[8];
            unpack8(__ldg(in + (((size_t)img * H + 2 * ho + dy) * W + 2 * wo + dx) * C8 + c), f);
#pragma unroll
            for (int j = 0; j < 8; ++j) acc[j] += f[j];
        }
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[j] *= 0.25f;
    out[idx] = pack8(acc);
}

// F.interpolate(scale_factor=2, mode="nearest") written into channels [coff, coff + C) of a wider NHWC buffer
__global__ void upsample_nearest2_kernel(const op_t* __restrict__ src, long long lds, int n_img, int Hs, int Ws, int C8,
                                         op_t* __restrict__ dst, long long ldd, int coff) {
    const int Hd = 2 * Hs, Wd = 2 * Ws;
    const long long total = (long long)n_img * Hd * Wd * C8;
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= total) return;
    const int c = (int)(idx % C8);
    const int wd = (int)((idx / C8) % Wd);
    const int hd = (int)((idx / ((long long)C8 * Wd)) % Hd);
    const int img = (int)(idx / ((long long)C8 * Wd * Hd));
    const uint4 v = __ldg(reinterpret_cast<const uint4*>(src + (((size_t)img * Hs + (hd >> 1)) * Ws + (wd >> 1)) * lds + c * 8));
    *reinterpret_cast<uint4*>(dst + (((size_t)img * Hd + hd) * Wd + wd) * ldd + coff + c * 8) = v;
}

// out = a + b (fp16, 8 per thread); b_f32 != null: out = a + b_f32[(row % period)] (fp32 table, e.g. position embedding)
__global__ void add_f16_kernel(const uint4* __restrict__ a, const uint4* __restrict__ b, const float* __restrict__ b_f32,
                               int C8, int period, uint4* __restrict__ out, long long total) {
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= total) return;
    float x[8], y[8];
    unpack8(__ldg(a + idx), x);
    if (b_f32 != nullptr) {
        const long long row = idx / C8;
        const float* p = b_f32 + ((row % period) * C8 + idx % C8) * 8;
#pragma unroll
        for (int j = 0; j < 8; ++j) y[j] = __ldg(p + j);
    } else {
        unpack8(__ldg(b + idx), y);
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) x[j] += y[j];
    out[idx] = pack8(x);
}

// rows outside the anchors' valid mask see a zero memory row (rtdetrv2_decoder.py:694): their enc_output.proj result is
// the bias.  x: fp32 [rows, D] GEMM output in LEVEL-MAJOR row order; one block per (invalid anchor, image).
__global__ void mask_invalid_rows_kernel(float* __restrict__ x, int D, const float* __restrict__ bias,
                                         const int* __restrict__ invalid, int n_invalid, RtLevels lv, int n_img) {
    const int a = invalid[blockIdx.x % n_invalid], img = blockIdx.x / n_invalid;
    const long long row = rt_anchor_row(lv, n_img, img, a);
    for (int c = threadIdx.x; c < D; c += blockDim.x) x[row * D + c] = bias[c];
}

// score[img][anchor] = max over classes of the encoder logits (level-major rows -> anchor-major scores)
__global__ void enc_scores_kernel(const float* __restrict__ logits, long long ldl, int C, RtLevels lv, int n_img,
                                  long long rows, float* __restrict__ scores) {
    const long long row = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (row >= rows) return;
    float m = -INFINITY;
    for (int c = 0; c < C; ++c) m = fmaxf(m, logits[row * ldl + c]);
    int img;
    const int a = rt_row_anchor_img(lv, n_img, row, &img);
    scores[(long long)img * lv.total + a] = m;
}

// torch.topk(scores, K) per image: one CTA sorts (score, anchor) keys with a bitonic network in shared memory.
// Order: descending score, ascending anchor among equal scores.  NP = power of two >= number of anchors.
__device__ __forceinline__ unsigned long long topk_key(float s, int a) {
    unsigned u = __float_as_uint(s);
    u = (u & 0x80000000u) ? ~u : (u | 0x80000000u);           // monotone map of the float order onto unsigned
    return ((unsigned long long)u << 32) | (unsigned)(0x7fffffff - a);
}
__global__ void topk_kernel(const float* __restrict__ scores, int L, int NP, int K, int* __restrict__ out_idx) {
    extern __shared__ unsigned long long keys[];
    const float* s = scores + (long long)blockIdx.x * L;
    for (int i = threadIdx.x; i < NP; i += blockDim.x) keys[i] = i < L ? topk_key(s[i], i) : 0ull;
    __syncthreads();
    for (int k = 2; k <= NP; k <<= 1)
        for (int j = k >> 1; j > 0; j >>= 1) {
            for (int i = threadIdx.x; i < NP; i += blockDim.x) {
                const int p = i ^ j;
                if (p > i) {
                    const unsigned long long a = keys[i], b = keys[p];
                    const bool desc = (i & k) == 0;              // descending blocks first: final order is descending
                    if (desc ? (a < b) : (a > b)) {
                        keys[i] = b;
                        keys[p] = a;
                    }
                }
            }
            __syncthreads();
        }
    for (int i = threadIdx.x; i < K; i += blockDim.x)
        out_idx[(long long)blockIdx.x * K + i] = 0x7fffffff - (int)(keys[i] & 0xffffffffu);
}

// The same result as topk_kernel for anchor counts whose full sort does not fit shared memory (the 960 cell detector:
// 18900 anchors).  One CTA of 1024 threads per image.  The scores stay in shared memory as 32-bit monotone keys; an
// MSB-first radix select (8 bits per pass) over the 48-bit key v = (score key << 16) | (0xffff - anchor) - the composite
// topk_key restricted to the bits that differ when L <= 65536 - finds the smallest prefix t such that exactly K keys have
// v >= t.  Those K keys are compacted into a next_pow2(K) buffer and bitonic-sorted (descending).  Every v is distinct,
// so the selected set and the order are fully determined; the passes over the anchor bits only run while scores tie.
constexpr int kSelThreads = 1024;
__device__ __forceinline__ unsigned score_key(float s) {
    const unsigned u = __float_as_uint(s);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);          // the map of topk_key
}
__global__ void __launch_bounds__(kSelThreads, 1)
topk_select_kernel(const float* __restrict__ scores, int L, int NK, int K, int* __restrict__ out_idx) {
    extern __shared__ unsigned long long sel_smem[];
    unsigned long long* sel = sel_smem;                                     // [NK] selected composite keys
    unsigned* hist = reinterpret_cast<unsigned*>(sel_smem + NK);            // [256]
    unsigned* skey = hist + 256;                                            // [L] score keys
    __shared__ unsigned long long s_prefix;    // digits chosen so far
    __shared__ unsigned s_need, s_cnt, s_n;    // keys still to take inside the prefix bucket, size of the chosen bucket
    const int tid = threadIdx.x, lane = tid & 31;
    const float* s = scores + (long long)blockIdx.x * L;
    for (int i = tid; i < L; i += kSelThreads) skey[i] = score_key(s[i]);
    if (tid == 0) {
        s_prefix = 0;
        s_need = K;
        s_n = 0;
    }
    int shift = 40;
    for (;; shift -= 8) {
        for (int i = tid; i < 256; i += kSelThreads) hist[i] = 0;
        __syncthreads();
        const unsigned long long prefix = s_prefix;
        for (int base = 0; base < L; base += kSelThreads) {
            const int i = base + tid;
            unsigned long long v = 0;
            bool in = false;
            if (i < L) {
                v = ((unsigned long long)skey[i] << 16) | (unsigned)(0xffff - i);
                in = (v >> (shift + 8)) == prefix;
            }
            const unsigned m = __ballot_sync(0xffffffffu, in);
            if (in) {
                // lanes with the same digit add once: quantised or blank-crop scores put thousands of keys in one bucket
                const unsigned d = (unsigned)(v >> shift) & 0xffu;
                const unsigned peers = __match_any_sync(m, d);
                if (lane == __ffs(peers) - 1) atomicAdd(&hist[d], __popc(peers));
            }
        }
        __syncthreads();
        if (tid < 32) {
            // lane l holds the bins 255 - 8 l down to 248 - 8 l; a scan over the lanes counts the keys in higher bins
            const unsigned need = s_need;
            unsigned c[8], sum = 0;
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                c[j] = hist[255 - 8 * lane - j];
                sum += c[j];
            }
            unsigned incl = sum;
#pragma unroll
            for (int off = 1; off < 32; off <<= 1) {
                const unsigned t = __shfl_up_sync(0xffffffffu, incl, off);
                if (lane >= off) incl += t;
            }
            unsigned above = incl - sum;
            if (above < need && need <= incl) {            // the bucket of the need-th largest key is in this lane
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    if (above + c[j] >= need) {
                        s_prefix = (prefix << 8) | (unsigned)(255 - 8 * lane - j);
                        s_need = need - above;
                        s_cnt = c[j];
                        break;
                    }
                    above += c[j];
                }
            }
        }
        __syncthreads();
        if (s_cnt == s_need) break;                        // the prefix buckets hold exactly K keys (at the latest at shift 0)
    }
    const unsigned long long thr = s_prefix << shift;
    for (int base = 0; base < L; base += kSelThreads) {
        const int i = base + tid;
        bool take = false;
        if (i < L) take = (((unsigned long long)skey[i] << 16) | (unsigned)(0xffff - i)) >= thr;
        const unsigned m = __ballot_sync(0xffffffffu, take);
        unsigned pos = 0;
        if (lane == 0 && m) pos = atomicAdd(&s_n, __popc(m));
        pos = __shfl_sync(0xffffffffu, pos, 0);
        if (take) sel[pos + __popc(m & ((1u << lane) - 1))] = ((unsigned long long)skey[i] << 32) | (unsigned)(0x7fffffff - i);
    }
    for (int i = K + tid; i < NK; i += kSelThreads) sel[i] = 0ull;        // below every real key
    __syncthreads();
    for (int k = 2; k <= NK; k <<= 1)
        for (int j = k >> 1; j > 0; j >>= 1) {
            for (int i = tid; i < NK; i += kSelThreads) {
                const int p = i ^ j;
                if (p > i) {
                    const unsigned long long a = sel[i], b = sel[p];
                    const bool desc = (i & k) == 0;
                    if (desc ? (a < b) : (a > b)) {
                        sel[i] = b;
                        sel[p] = a;
                    }
                }
            }
            __syncthreads();
        }
    for (int i = tid; i < K; i += kSelThreads)
        out_idx[(long long)blockIdx.x * K + i] = 0x7fffffff - (int)(sel[i] & 0xffffffffu);
}

// decoder start: target rows = output_memory[top-k rows] (fp32 + fp16), anchors of the selected positions
__global__ void gather_queries_kernel(const float* __restrict__ om, int D, const int* __restrict__ idx, int K, RtLevels lv,
                                      int n_img, float* __restrict__ tgt, op_t* __restrict__ tgt16,
                                      const float* __restrict__ anchors, float* __restrict__ anchor_sel) {
    const int q = blockIdx.x;                    // img * K + j
    const int img = q / K;
    const int a = idx[q];
    const long long row = rt_anchor_row(lv, n_img, img, a);
    for (int c = threadIdx.x; c < D; c += blockDim.x) {
        const float v = om[row * D + c];
        tgt[(long long)q * D + c] = v;
        tgt16[(long long)q * D + c] = f2op(v);
    }
    if (threadIdx.x < 4) anchor_sel[q * 4 + threadIdx.x] = anchors[a * 4 + threadIdx.x];
}

__device__ __forceinline__ float sigmoidf_(float x) { return 1.f / (1.f + expf(-x)); }
__device__ __forceinline__ float inv_sigmoid(float x) {
    x = fminf(fmaxf(x, 0.f), 1.f);
    return logf(fmaxf(x, 1e-5f) / fmaxf(1.f - x, 1e-5f));
}

// ref = sigmoid(delta + base): base = the selected anchors (logit space, start) or inverse_sigmoid(ref) (refinement)
__global__ void ref_update_kernel(const float* __restrict__ delta, long long ldd, const float* __restrict__ anchor_sel,
                                  float* __restrict__ ref, int n) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n * 4) return;
    const float base = anchor_sel != nullptr ? anchor_sel[i] : inv_sigmoid(ref[i]);
    ref[i] = sigmoidf_(delta[(long long)(i >> 2) * ldd + (i & 3)] + base);
}

// first layer of query_pos_head: relu(W [H1, 4] ref + b) -> fp16 [rows, H1] (K = 4 is no GEMM)
__global__ void qpos_l0_kernel(const float* __restrict__ ref, const float* __restrict__ W, const float* __restrict__ b,
                               int H1, op_t* __restrict__ out, long long total) {
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= total) return;
    const long long row = idx / H1;
    const int j = (int)(idx % H1);
    const float4 r = *reinterpret_cast<const float4*>(ref + row * 4);
    const float4 w = *reinterpret_cast<const float4*>(W + j * 4);
    out[idx] = f2op(fmaxf(b[j] + w.x * r.x + w.y * r.y + w.z * r.z + w.w * r.w, 0.f));
}

// Multi-scale deformable attention core (rtdetrv2_decoder.py:306-388, method "default") for 4-d reference boxes
// (:197-207).  One warp per (query, head), lane = channel of the head (head_dim 32).
//   ow: fp32 [rows, ldo] = sampling offsets (heads * P * 2) followed by attention logits (heads * P) of the query
//   value: fp16 level-major [.., ldv], the head's 32 channels at column voff + head * 32
//   loc = ref.xy + off * (1 / points of the level) * ref.wh * 0.5; bilinear, zero padding, align_corners = False
template <int P>
__global__ void deform_attn_kernel(const float* __restrict__ ow, long long ldo, const float* __restrict__ ref,
                                   const op_t* __restrict__ value, long long ldv, int voff, RtLevels lv, int n_img, int K,
                                   int heads, float offset_scale, op_t* __restrict__ out, long long ldout, int rows) {
    const int warp = (int)(((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5);
    const int lane = threadIdx.x & 31;
    if (warp >= rows * heads) return;
    const int row = warp / heads, head = warp - row * heads;
    const int img = row / K;
    const float* o = ow + (long long)row * ldo;
    // softmax over the P attention logits of this head (every lane computes it: P is 12)
    float wts[P];
    float mx = -INFINITY;
#pragma unroll
    for (int p = 0; p < P; ++p) {
        wts[p] = o[heads * P * 2 + head * P + p];
        mx = fmaxf(mx, wts[p]);
    }
    float sum = 0.f;
#pragma unroll
    for (int p = 0; p < P; ++p) {
        wts[p] = expf(wts[p] - mx);
        sum += wts[p];
    }
    const float inv = 1.f / sum;
    const float4 r = *reinterpret_cast<const float4*>(ref + (long long)row * 4);
    float acc = 0.f;
    int p = 0;
#pragma unroll
    for (int l = 0; l < RtLevels::kMax; ++l) {
        if (l >= lv.n) break;
        const int H = lv.h[l], W = lv.w[l], np = lv.points[l];
        const op_t* vbase = value + ((long long)lv.off[l] * n_img + (long long)img * H * W) * ldv + voff + head * 32 + lane;
        const float pscale = 1.f / (float)np;
        for (int k = 0; k < np; ++k, ++p) {
            const float ox = o[(head * P + p) * 2 + 0], oy = o[(head * P + p) * 2 + 1];
            const float lx = r.x + ox * pscale * r.z * offset_scale, ly = r.y + oy * pscale * r.w * offset_scale;
            // grid_sample(align_corners=False): pixel coordinate = ((2 loc - 1) + 1) * size / 2 - 0.5 = loc * size - 0.5
            const float gx = 2.f * lx - 1.f, gy = 2.f * ly - 1.f;
            const float x = ((gx + 1.f) * W - 1.f) * 0.5f, y = ((gy + 1.f) * H - 1.f) * 0.5f;
            const float xf = floorf(x), yf = floorf(y);
            const int x0 = (int)xf, y0 = (int)yf;
            const float ax = x - xf, ay = y - yf;
            float v = 0.f;
            if (y0 >= 0 && y0 < H) {
                if (x0 >= 0 && x0 < W) v += (1.f - ay) * (1.f - ax) * op2f(vbase[((long long)y0 * W + x0) * ldv]);
                if (x0 + 1 >= 0 && x0 + 1 < W) v += (1.f - ay) * ax * op2f(vbase[((long long)y0 * W + x0 + 1) * ldv]);
            }
            if (y0 + 1 >= 0 && y0 + 1 < H) {
                if (x0 >= 0 && x0 < W) v += ay * (1.f - ax) * op2f(vbase[((long long)(y0 + 1) * W + x0) * ldv]);
                if (x0 + 1 >= 0 && x0 + 1 < W) v += ay * ax * op2f(vbase[((long long)(y0 + 1) * W + x0 + 1) * ldv]);
            }
            acc += wts[p] * inv * v;
        }
    }
    out[(long long)row * ldout + head * 32 + lane] = f2op(acc);
}

// fp32 [rows, ld] -> packed [rows, C] fp32 (the C ABI's outputs)
__global__ void copy_cols_kernel(const float* __restrict__ src, long long ld, int C, float* __restrict__ dst, long long total) {
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= total) return;
    dst[idx] = src[(idx / C) * ld + idx % C];
}

inline unsigned blocks_for(long long total, int threads = 256) { return (unsigned)((total + threads - 1) / threads); }

}  // namespace

int launch_rt_pack_input(const float* src, int n_img, int H, int W, void* dst, cudaStream_t st) {
    const long long total = (long long)n_img * H * W * 8;
    pack_input_kernel<<<blocks_for(total), 256, 0, st>>>(src, n_img, H, W, reinterpret_cast<uint4*>(dst));
    count_launch();
    return cudaGetLastError() != cudaSuccess;
}

int launch_rt_avgpool2(const void* in, void* out, int n_img, int H, int W, int C, cudaStream_t st) {
    if ((H | W) & 1 || C % 8) {
        set_error("avgpool2: H, W must be even and C a multiple of 8 (got %dx%dx%d)", H, W, C);
        return 1;
    }
    const long long total = (long long)n_img * (H / 2) * (W / 2) * (C / 8);
    avgpool2_kernel<<<blocks_for(total), 256, 0, st>>>(reinterpret_cast<const uint4*>(in), reinterpret_cast<uint4*>(out),
                                                       n_img, H, W, C / 8);
    count_launch();
    return cudaGetLastError() != cudaSuccess;
}

int launch_rt_upsample_nearest2(const void* src, long long lds, int n_img, int Hs, int Ws, int C, void* dst, long long ldd,
                                int coff, cudaStream_t st) {
    const long long total = (long long)n_img * 4 * Hs * Ws * (C / 8);
    upsample_nearest2_kernel<<<blocks_for(total), 256, 0, st>>>(reinterpret_cast<const op_t*>(src), lds, n_img, Hs, Ws, C / 8,
                                                                reinterpret_cast<op_t*>(dst), ldd, coff);
    count_launch();
    return cudaGetLastError() != cudaSuccess;
}

int launch_rt_add(const void* a, const void* b, const float* b_f32, int C, int period, void* out, long long rows,
                  cudaStream_t st) {
    const long long total = rows * (C / 8);
    add_f16_kernel<<<blocks_for(total), 256, 0, st>>>(reinterpret_cast<const uint4*>(a), reinterpret_cast<const uint4*>(b),
                                                      b_f32, C / 8, period > 0 ? period : 1,
                                                      reinterpret_cast<uint4*>(out), total);
    count_launch();
    return cudaGetLastError() != cudaSuccess;
}

int launch_rt_mask_invalid(float* x, int D, const float* bias, const int* invalid, int n_invalid, const RtLevels& lv,
                           int n_img, cudaStream_t st) {
    if (n_invalid <= 0) return 0;
    mask_invalid_rows_kernel<<<n_invalid * n_img, 128, 0, st>>>(x, D, bias, invalid, n_invalid, lv, n_img);
    count_launch();
    return cudaGetLastError() != cudaSuccess;
}

int launch_rt_enc_scores(const float* logits, long long ldl, int C, const RtLevels& lv, int n_img, float* scores,
                         cudaStream_t st) {
    const long long rows = (long long)lv.total * n_img;
    enc_scores_kernel<<<blocks_for(rows), 256, 0, st>>>(logits, ldl, C, lv, n_img, rows, scores);
    count_launch();
    return cudaGetLastError() != cudaSuccess;
}

int launch_rt_topk(const float* scores, int n_img, int L, int K, int* out_idx, cudaStream_t st) {
    int NP = 1;
    while (NP < L) NP <<= 1;
    const size_t smem = (size_t)NP * sizeof(unsigned long long);
    if (smem > (size_t)kTopkSmemBytes) return launch_rt_topk_select(scores, n_img, L, K, out_idx, st);
    static unsigned long long attr_done = 0;   // per device
    if (first_launch_on_device(&attr_done)) {
        if (cudaFuncSetAttribute(topk_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kTopkSmemBytes) != cudaSuccess) {
            set_error("topk: cannot raise the shared memory limit");
            return 1;
        }
    }
    if (K > L) {
        set_error("topk: %d candidates / k = %d unsupported", L, K);
        return 1;
    }
    topk_kernel<<<n_img, 1024, smem, st>>>(scores, L, NP, K, out_idx);
    count_launch();
    return cudaGetLastError() != cudaSuccess;
}

int launch_rt_topk_select(const float* scores, int n_img, int L, int K, int* out_idx, cudaStream_t st) {
    if (L < 1 || L > kTopkSelectMaxL || K < 1 || K > kTopkSelectMaxK || K > L) {
        set_error("topk: %d candidates / k = %d unsupported (radix select: 1 <= k <= min(%d, candidates), candidates <= %d)",
                  L, K, kTopkSelectMaxK, kTopkSelectMaxL);
        return 1;
    }
    int NK = 1;
    while (NK < K) NK <<= 1;
    const size_t smem = (size_t)NK * sizeof(unsigned long long) + 256 * sizeof(unsigned) + (size_t)L * sizeof(unsigned);
    static unsigned long long attr_done = 0;   // per device
    if (first_launch_on_device(&attr_done)) {
        if (cudaFuncSetAttribute(topk_select_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kTopkSmemBytes) !=
            cudaSuccess) {
            set_error("topk: cannot raise the shared memory limit");
            return 1;
        }
    }
    topk_select_kernel<<<n_img, kSelThreads, smem, st>>>(scores, L, NK, K, out_idx);
    count_launch();
    return cudaGetLastError() != cudaSuccess;
}

int launch_rt_gather_queries(const float* om, int D, const int* idx, int K, const RtLevels& lv, int n_img, float* tgt,
                             void* tgt16, const float* anchors, float* anchor_sel, cudaStream_t st) {
    gather_queries_kernel<<<n_img * K, 128, 0, st>>>(om, D, idx, K, lv, n_img, tgt, reinterpret_cast<op_t*>(tgt16),
                                                     anchors, anchor_sel);
    count_launch();
    return cudaGetLastError() != cudaSuccess;
}

int launch_rt_ref_update(const float* delta, long long ldd, const float* anchor_sel, float* ref, int n, cudaStream_t st) {
    ref_update_kernel<<<blocks_for((long long)n * 4, 128), 128, 0, st>>>(delta, ldd, anchor_sel, ref, n);
    count_launch();
    return cudaGetLastError() != cudaSuccess;
}

int launch_rt_qpos_l0(const float* ref, const float* W, const float* b, int H1, void* out, int rows, cudaStream_t st) {
    const long long total = (long long)rows * H1;
    qpos_l0_kernel<<<blocks_for(total), 256, 0, st>>>(ref, W, b, H1, reinterpret_cast<op_t*>(out), total);
    count_launch();
    return cudaGetLastError() != cudaSuccess;
}

int launch_rt_deform_attn(const float* ow, long long ldo, const float* ref, const void* value, long long ldv, int voff,
                          const RtLevels& lv, int n_img, int K, int heads, int head_dim, float offset_scale, void* out,
                          long long ldout, cudaStream_t st) {
    int P = 0;
    for (int l = 0; l < lv.n; ++l) P += lv.points[l];
    if (head_dim != 32 || P != 12) {
        set_error("deformable attention: head_dim %d / %d points per head unsupported (32 / 12)", head_dim, P);
        return 1;
    }
    const int rows = n_img * K;
    const long long threads = (long long)rows * heads * 32;
    deform_attn_kernel<12><<<blocks_for(threads), 256, 0, st>>>(ow, ldo, ref, reinterpret_cast<const op_t*>(value), ldv,
                                                                voff, lv, n_img, K, heads, offset_scale,
                                                                reinterpret_cast<op_t*>(out), ldout, rows);
    count_launch();
    return cudaGetLastError() != cudaSuccess;
}

int launch_rt_copy_cols(const float* src, long long ld, int C, float* dst, long long rows, cudaStream_t st) {
    copy_cols_kernel<<<blocks_for(rows * C), 256, 0, st>>>(src, ld, C, dst, rows * C);
    count_launch();
    return cudaGetLastError() != cudaSuccess;
}

}  // namespace ytk
