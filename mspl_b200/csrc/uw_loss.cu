// K4 (fused rectified uncertainty-weighted CE forward+backward), K0 (get_output's softmax + KLD maps) and the
// generic forms behind the reference's two nn.Modules (PixelwiseKLD, UncertaintyWeightedSegmentationLoss).
//
// Closed forms (verified against reference autograd in fp64, tests/test_oracle_vs_reference.py):
//   per pixel  z = m + a/2, q = softmax(z), p1 = softmax(m), p2 = softmax(a), D = sum_k p1_k (log p1_k - log p2_k),
//              ce = w_t * (-log q_t),  N = number of pixels in the mean
//   L        = (alpha/N) sum ce e^{-D} + (1/N) sum D                       uest_seg_multi_os.py:1020-1023
//   dL/dz_k  = (alpha/N) e^{-D} w_t (q_k - [k==t])
//   g_D      = (1 - alpha ce e^{-D}) / N
//   dL/dm_k  = dL/dz_k + g_D p1_k (log p1_k - log p2_k - D)
//   dL/da_k  = dL/dz_k / 2 + g_D (p2_k - p1_k)
#include <algorithm>
#include <cstring>

#include "pixel_math.cuh"
#include "bilinear.cuh"

namespace mspl {

constexpr int kLossThreads = 256;
constexpr int kMaxLossBlocks = 2048;

struct LossWorkspace {            // caller-zeroed once; every launch leaves `ticket` at 0 again
    unsigned int ticket;
    unsigned int pad[3];
    double partial[kMaxLossBlocks][2];
};

// Deterministic two-value reduction: per-thread doubles -> warp shuffle -> block -> per-block slot; the last block
// to finish adds the slots in index order and writes the means.  No floating-point atomics anywhere.
template <int NOUT, int NT = kLossThreads>
MSPL_DEVINL void finish_loss(double s0, double s1, LossWorkspace* ws, double inv_n, float alpha, float* out) {
    __shared__ double s_part[NT / 32][2];
    __shared__ bool s_last;
    s0 = warp_sum(s0);
    s1 = warp_sum(s1);
    if ((threadIdx.x & 31) == 0) { s_part[threadIdx.x >> 5][0] = s0; s_part[threadIdx.x >> 5][1] = s1; }
    __syncthreads();
    if (threadIdx.x == 0) {
        double a = 0, b = 0;
        for (int w = 0; w < NT / 32; ++w) { a += s_part[w][0]; b += s_part[w][1]; }
        ws->partial[blockIdx.x][0] = a;
        ws->partial[blockIdx.x][1] = b;
        __threadfence();
        s_last = atomicAdd(&ws->ticket, 1u) == gridDim.x - 1;
    }
    __syncthreads();
    if (!s_last) return;
    __threadfence();
    double a = 0, b = 0;
    for (int i = threadIdx.x; i < (int)gridDim.x; i += NT) {   // fixed assignment -> fixed order
        a += __ldcg(&ws->partial[i][0]);
        b += __ldcg(&ws->partial[i][1]);
    }
    a = warp_sum(a);
    b = warp_sum(b);
    __syncthreads();
    if ((threadIdx.x & 31) == 0) { s_part[threadIdx.x >> 5][0] = a; s_part[threadIdx.x >> 5][1] = b; }
    __syncthreads();
    if (threadIdx.x == 0) {
        a = b = 0;
        for (int w = 0; w < NT / 32; ++w) { a += s_part[w][0]; b += s_part[w][1]; }
        const double ce_mean = a * inv_n, kld_mean = b * inv_n;
        if (NOUT == 3) {
            out[0] = (float)((double)alpha * ce_mean + kld_mean);
            out[1] = (float)ce_mean;
            out[2] = (float)kld_mean;
        } else {
            out[0] = (float)ce_mean;
        }
        ws->ticket = 0;
    }
}

// One pixel of K4 (closed forms in the file header): l = w_t ce e^{-D}, D = KL(softmax m || softmax a), and for BWD the
// gradients of (gscale/N) * (alpha * sum l + sum D) w.r.t. the K main and aux logits.
template <int K, bool BWD>
MSPL_DEVINL void uw_ce_pixel(const float (&m)[K], const float (&a)[K], long long t, const float* s_w, float alpha, float gscale,
                             float inv_nf, float& l, float& D, float (&gm)[K], float (&ga)[K]) {
    float z[K], Mm = -INFINITY, Ma = -INFINITY, Mz = -INFINITY;
#pragma unroll
    for (int k = 0; k < K; ++k) {
        z[k] = fmaf(0.5f, a[k], m[k]);
        Mm = fmaxf(Mm, m[k]); Ma = fmaxf(Ma, a[k]); Mz = fmaxf(Mz, z[k]);
    }
    float em[K], ea[K], ez[K], Sm = 0.f, Sa = 0.f, Sz = 0.f;
#pragma unroll
    for (int k = 0; k < K; ++k) {
        em[k] = exp_neg(m[k] - Mm); ea[k] = exp_neg(a[k] - Ma); ez[k] = exp_neg(z[k] - Mz);
        Sm += em[k]; Sa += ea[k]; Sz += ez[k];
    }
    const float rSm = rcp_fast(Sm), rSa = rcp_fast(Sa), rSz = rcp_fast(Sz);
    const float lRatio = log_fast(Sm * rSa), lSz = log_fast(Sz);     // log Sm - log Sa, log Sz
    float dl[K];                             // dl_k = log p1_k - log p2_k
    D = 0.f;
#pragma unroll
    for (int k = 0; k < K; ++k) {
        dl[k] = ((m[k] - Mm) - (a[k] - Ma)) - lRatio;
        D = fmaf(em[k] * rSm, dl[k], D);
    }
    const int ti = (int)t;
    const bool valid = t >= 0 && t < K;
    float wt = 0.f, zt = Mz;
#pragma unroll
    for (int k = 0; k < K; ++k) {
        wt = (valid && ti == k) ? s_w[k] : wt;
        zt = (valid && ti == k) ? z[k] : zt;
    }
    const float ce = wt * (lSz - (zt - Mz));
    const float eD = exp_neg(-D);
    l = ce * eD;
    if (BWD) {
        const float coef = gscale * alpha * inv_nf * eD * wt;
        const float gD = gscale * inv_nf * (1.0f - alpha * l);
#pragma unroll
        for (int k = 0; k < K; ++k) {
            const float p1 = em[k] * rSm, p2 = ea[k] * rSa, q = ez[k] * rSz;
            const float dz = coef * (q - ((valid && ti == k) ? 1.0f : 0.0f));
            gm[k] = fmaf(gD, p1 * (dl[k] - D), dz);
            ga[k] = fmaf(gD, p2 - p1, 0.5f * dz);
        }
    }
}

// ---- K4 ------------------------------------------------------------------------------------------------
// Targets of P consecutive pixels as class indices: int64 (what torch's gather wants, the reference's format) or uint8 (the
// format the label maps are generated and stored in: 1 B/pixel instead of 8).
template <int P> MSPL_DEVINL void load_targets(const int64_t* p, long long (&t)[P]) {
    if (P == 4) {
        const longlong2 t0 = __ldcs(reinterpret_cast<const longlong2*>(p));
        const longlong2 t1 = __ldcs(reinterpret_cast<const longlong2*>(p) + 1);
        t[0] = t0.x; t[1] = t0.y; t[P > 2 ? 2 : 0] = t1.x; t[P > 3 ? 3 : 0] = t1.y;
    } else if (P == 2) {
        const longlong2 t0 = __ldcs(reinterpret_cast<const longlong2*>(p));
        t[0] = t0.x; t[P > 1 ? 1 : 0] = t0.y;
    } else {
#pragma unroll
        for (int i = 0; i < P; ++i) t[i] = __ldcs(p + i);
    }
}
template <int P> MSPL_DEVINL void load_targets(const uint8_t* p, long long (&t)[P]) {
    if (P == 4) {
        const uchar4 v = __ldcs(reinterpret_cast<const uchar4*>(p));
        t[0] = v.x; t[1] = v.y; t[P > 2 ? 2 : 0] = v.z; t[P > 3 ? 3 : 0] = v.w;
    } else if (P == 2) {
        const uchar2 v = __ldcs(reinterpret_cast<const uchar2*>(p));
        t[0] = v.x; t[P > 1 ? 1 : 0] = v.y;
    } else {
#pragma unroll
        for (int i = 0; i < P; ++i) t[i] = __ldcs(p + i);
    }
}

// Three resident CTAs per SM: without the bound ptxas spends 126 registers on the P=2 backward (2 CTAs/SM); capped at 85 it
// needs 80, spills nothing, and the third CTA's loads in flight are worth +6.5 % (profiles/r01_loss_variants.txt).  K = 7, 8
// would spill under that cap and keep two CTAs.
// ---- MIOU.get_iou counts folded into K4 (the training loop calls it on the very tensors the loss reads,
// uest_seg_multi_os.py:1032: `inter, union = miou_class.get_iou(pred, labels)`) -------------------------------------------
// Semantics of utilities/metrics/segmentation_miou.py:13-44 as in miou.cu: pred = first-max argmax of the MAIN logits, both
// sides cast to uint8 and shifted by one, pixels with shifted target 0 dropped, classes outside [1, K] not counted.
// Per-thread counts live in shared memory, one word per class and thread ([K][threads]: conflict-free), three 10-bit fields
// [inter | pred | mask] per word, folded into the CTA's totals before a field can overflow: no atomics, no warp votes and
// no registers in the pixel loop (the P=2 backward has none to spare under its 80-register occupancy bound).
constexpr int kIouFieldBits = 10;
constexpr int kIouFlushPixels = (1 << kIouFieldBits) - 8;

template <int K>
MSPL_DEVINL void iou_tally(const float (&m)[K], long long t, uint32_t* my_cnt) {      // my_cnt = s_cnt + threadIdx.x
    int am = 0;
    float best = m[0];
#pragma unroll
    for (int k = 1; k < K; ++k) {
        am = (m[k] > best) ? k : am;          // strict >: first maximal index, as torch.max(output, 1)
        best = fmaxf(best, m[k]);
    }
    const uint32_t ts = ((uint32_t)t + 1u) & 0xffu;            // ByteTensor cast, += 1 "so that 255 is 0"
    if (ts == 0) return;                                       // pred * (target > 0): nothing to count for this pixel
    const uint32_t ps = (uint32_t)am + 1u;                     // always in [1, K]
    my_cnt[(ps - 1) * kLossThreads] += 1u << kIouFieldBits;
    if (ts <= (uint32_t)K) my_cnt[(ts - 1) * kLossThreads] += 1u + (ps == ts ? (1u << (2 * kIouFieldBits)) : 0u);
}

// Unpack this thread's fields, add them to the CTA's totals s_iou[3][K] (stored [inter | pred | mask]) and clear.
// WARP: every lane of the warp is here (the flush after the pixel loop), so reduce over the warp first; otherwise (the rare
// mid-loop flush, once per ~1,000 pixels of a thread) each thread adds its own fields and no convergence is assumed.
template <int K, bool WARP>
MSPL_DEVINL void iou_flush(uint32_t* my_cnt, uint32_t* s_iou) {
    constexpr uint32_t kMask = (1u << kIouFieldBits) - 1u;
#pragma unroll
    for (int k = 0; k < K; ++k) {
        const uint32_t word = my_cnt[k * kLossThreads];
        my_cnt[k * kLossThreads] = 0;
#pragma unroll
        for (int f = 0; f < 3; ++f) {
            uint32_t v = (word >> (f * kIouFieldBits)) & kMask;       // f: 0 mask, 1 pred, 2 inter
            if (WARP) v = __reduce_add_sync(0xffffffffu, v);
            if ((!WARP || (threadIdx.x & 31) == 0) && v) atomicAdd(&s_iou[(2 - f) * K + k], v);
        }
    }
}

#ifndef MSPL_UWCE_MINB
#define MSPL_UWCE_MINB 3
#endif
#ifndef MSPL_UWCE_BWD_P
#define MSPL_UWCE_BWD_P 2
#endif
// The body of K4.  LT: logit and gradient element type, float or the __half / __nv_bfloat16 logits of an autocast forward;
// every per-pixel operation is on the fp32 values either way.
template <int P, int K, bool BWD, typename TT, bool IOU, typename LT>
MSPL_DEVINL void uw_ce_fused(const LT* __restrict__ main_l, const LT* __restrict__ aux_l, const TT* __restrict__ target,
                             const float* __restrict__ cw, int64_t n_img, int64_t hw, float alpha, double inv_n, float gscale,
                             float* __restrict__ out3, LT* __restrict__ d_main, LT* __restrict__ d_aux, LossWorkspace* ws,
                             unsigned long long* __restrict__ iou_counts) {
    __shared__ float s_w[K];
    __shared__ uint32_t s_iou[3 * K];
    __shared__ uint32_t s_cnt[IOU ? K * kLossThreads : 1];
    uint32_t* const my_cnt = s_cnt + (IOU ? threadIdx.x : 0);
    if (threadIdx.x < K) s_w[threadIdx.x] = cw[threadIdx.x];
    if (IOU) {
        if (threadIdx.x < 3 * K) s_iou[threadIdx.x] = 0;
#pragma unroll
        for (int k = 0; k < K; ++k) my_cnt[k * kLossThreads] = 0;
    }
    int iou_pixels = 0;
    __syncthreads();
    const int64_t gpi = hw / P, n_groups = n_img * gpi;
    const float inv_nf = (float)inv_n;
    double acc_ce = 0, acc_d = 0;
    for (int64_t g = blockIdx.x * (int64_t)kLossThreads + threadIdx.x; g < n_groups; g += (int64_t)gridDim.x * kLossThreads) {
        const int64_t n = g / gpi, off = (g - n * gpi) * P;
        const int64_t base = n * K * hw + off;
        float m[K][P], a[K][P];
        long long t[P];
#pragma unroll
        for (int k = 0; k < K; ++k) LogitVec<LT, P>::load(main_l + base + k * hw, m[k]);
#pragma unroll
        for (int k = 0; k < K; ++k) LogitVec<LT, P>::load(aux_l + base + k * hw, a[k]);
        load_targets<P>(target + n * hw + off, t);
        float gm[K][P], ga[K][P];
        float ce_sum = 0.f, d_sum = 0.f;
#pragma unroll
        for (int p = 0; p < P; ++p) {
            float mp[K], ap[K], gmp[K], gap[K], l, D;
#pragma unroll
            for (int k = 0; k < K; ++k) { mp[k] = m[k][p]; ap[k] = a[k][p]; }
            uw_ce_pixel<K, BWD>(mp, ap, t[p], s_w, alpha, gscale, inv_nf, l, D, gmp, gap);
            if (IOU) iou_tally<K>(mp, t[p], my_cnt);
            ce_sum += l;
            d_sum += D;
            if (BWD) {
#pragma unroll
                for (int k = 0; k < K; ++k) { gm[k][p] = gmp[k]; ga[k][p] = gap[k]; }
            }
        }
        acc_ce += (double)ce_sum;
        acc_d += (double)d_sum;
        if (BWD) {
#pragma unroll
            for (int k = 0; k < K; ++k) LogitVec<LT, P>::store(d_main + base + k * hw, gm[k]);
#pragma unroll
            for (int k = 0; k < K; ++k) LogitVec<LT, P>::store(d_aux + base + k * hw, ga[k]);
        }
        if (IOU) {
            iou_pixels += P;
            if (iou_pixels >= kIouFlushPixels) {      // a field holds < 2^10 pixels
                iou_flush<K, false>(my_cnt, s_iou);
                iou_pixels = 0;
            }
        }
    }
    if (IOU) {
        iou_flush<K, true>(my_cnt, s_iou);
        __syncthreads();
        if (threadIdx.x < 3 * K && s_iou[threadIdx.x]) atomicAdd(iou_counts + threadIdx.x, (unsigned long long)s_iou[threadIdx.x]);
    }
    finish_loss<3>(acc_ce, acc_d, ws, inv_n, alpha, out3);
}

template <int P, int K, bool BWD, typename TT, bool IOU>
__global__ void __launch_bounds__(kLossThreads, (K <= 6 ? MSPL_UWCE_MINB : 2)) uw_ce_fused_kernel(const float* __restrict__ main_l, const float* __restrict__ aux_l,
                                                                   const TT* __restrict__ target, const float* __restrict__ cw,
                                                                   int64_t n_img, int64_t hw, float alpha, double inv_n, float gscale,
                                                                   float* __restrict__ out3, float* __restrict__ d_main,
                                                                   float* __restrict__ d_aux, LossWorkspace* ws,
                                                                   unsigned long long* __restrict__ iou_counts) {
    uw_ce_fused<P, K, BWD, TT, IOU, float>(main_l, aux_l, target, cw, n_img, hw, alpha, inv_n, gscale, out3, d_main, d_aux, ws,
                                           iou_counts);
}

// K4 on fp16 / bf16 logits.  gscale_dev (may be NULL): a device scalar the gradients are also scaled by -- the upstream
// gradient of the autograd backward (a GradScaler's loss scale) -- applied BEFORE the rounding to LT, since gradient terms
// far below the fp16 subnormal range only become representable after it.
template <int P, int K, bool BWD, typename TT, bool IOU, typename LT>
__global__ void __launch_bounds__(kLossThreads, (K <= 6 ? MSPL_UWCE_MINB : 2)) uw_ce_fused_half_kernel(const LT* __restrict__ main_l, const LT* __restrict__ aux_l,
                                                                   const TT* __restrict__ target, const float* __restrict__ cw,
                                                                   int64_t n_img, int64_t hw, float alpha, double inv_n, float gscale,
                                                                   float* __restrict__ out3, LT* __restrict__ d_main,
                                                                   LT* __restrict__ d_aux, LossWorkspace* ws,
                                                                   unsigned long long* __restrict__ iou_counts,
                                                                   const float* __restrict__ gscale_dev) {
    if (BWD && gscale_dev) gscale *= __ldg(gscale_dev);
    uw_ce_fused<P, K, BWD, TT, IOU, LT>(main_l, aux_l, target, cw, n_img, hw, alpha, inv_n, gscale, out3, d_main, d_aux, ws,
                                        iou_counts);
}

}  // namespace mspl

#include "uw_loss_lowres.cuh"

namespace mspl {

// ---- generic runtime-C helpers (compat paths; logits are re-read from L1/L2, HBM sees them once) -------------
// softmax statistics of one logit vector per pixel: M = max, S = sum e^{x-M}
template <int P>
MSPL_DEVINL void stats1(const float* __restrict__ px, int C, int64_t hw, float (&M)[P], float (&S)[P]) {
#pragma unroll
    for (int p = 0; p < P; ++p) { M[p] = -INFINITY; S[p] = 0.f; }
    for (int c = 0; c < C; ++c) {
        float v[P];
        PixVec<P>::load(px + c * hw, v);
#pragma unroll
        for (int p = 0; p < P; ++p) M[p] = fmaxf(M[p], v[p]);
    }
    for (int c = 0; c < C; ++c) {
        float v[P];
        PixVec<P>::load(px + c * hw, v);
#pragma unroll
        for (int p = 0; p < P; ++p) S[p] += exp_neg(v[p] - M[p]);
    }
}

// D = KL(softmax(x1) || softmax(x2)) with the pieces the backward needs.
template <int P>
struct KldStats { float M1[P], S1[P], M2[P], S2[P], D[P]; };

template <int P>
MSPL_DEVINL void kld_stats(const float* __restrict__ p1, const float* __restrict__ p2, int C, int64_t hw, KldStats<P>& k) {
    stats1<P>(p1, C, hw, k.M1, k.S1);
    stats1<P>(p2, C, hw, k.M2, k.S2);
    float l1[P], l2[P], r1[P];
#pragma unroll
    for (int p = 0; p < P; ++p) { l1[p] = logf(k.S1[p]); l2[p] = logf(k.S2[p]); r1[p] = 1.0f / k.S1[p]; k.D[p] = 0.f; }
    for (int c = 0; c < C; ++c) {
        float x[P], y[P];
        PixVec<P>::load(p1 + c * hw, x);
        PixVec<P>::load(p2 + c * hw, y);
#pragma unroll
        for (int p = 0; p < P; ++p) {
            const float t1 = x[p] - k.M1[p];
            k.D[p] = fmaf(exp_neg(t1) * r1[p], (t1 - l1[p]) - ((y[p] - k.M2[p]) - l2[p]), k.D[p]);
        }
    }
}

// K0: prob = softmax(main + aux/2), kld = KL(softmax(main)||softmax(aux))        uest_seg_multi_os.py:687-691
template <int P>
__global__ void __launch_bounds__(256) softmax_kld_kernel(const float* __restrict__ main_l, const float* __restrict__ aux_l, int64_t n_img,
                                                          int C, int64_t hw, float* __restrict__ prob, float* __restrict__ kld) {
    const int64_t gpi = hw / P, n_groups = n_img * gpi;
    for (int64_t g = blockIdx.x * 256ll + threadIdx.x; g < n_groups; g += (int64_t)gridDim.x * 256) {
        const int64_t n = g / gpi, off = (g - n * gpi) * P;
        const float* pm = main_l + n * C * hw + off;
        const float* pa = aux_l + n * C * hw + off;
        if (kld) {
            KldStats<P> ks;
            kld_stats<P>(pm, pa, C, hw, ks);
            PixVec<P>::store(kld + n * hw + off, ks.D);
        }
        if (prob) {
            float M[P], S[P], r[P];
#pragma unroll
            for (int p = 0; p < P; ++p) { M[p] = -INFINITY; S[p] = 0.f; }
            for (int c = 0; c < C; ++c) {
                float x[P], y[P];
                PixVec<P>::load(pm + c * hw, x);
                PixVec<P>::load(pa + c * hw, y);
#pragma unroll
                for (int p = 0; p < P; ++p) M[p] = fmaxf(M[p], fmaf(0.5f, y[p], x[p]));
            }
            for (int c = 0; c < C; ++c) {
                float x[P], y[P];
                PixVec<P>::load(pm + c * hw, x);
                PixVec<P>::load(pa + c * hw, y);
#pragma unroll
                for (int p = 0; p < P; ++p) S[p] += exp_neg(fmaf(0.5f, y[p], x[p]) - M[p]);
            }
#pragma unroll
            for (int p = 0; p < P; ++p) r[p] = 1.0f / S[p];
            for (int c = 0; c < C; ++c) {
                float x[P], y[P], o[P];
                PixVec<P>::load(pm + c * hw, x);
                PixVec<P>::load(pa + c * hw, y);
#pragma unroll
                for (int p = 0; p < P; ++p) o[p] = exp_neg(fmaf(0.5f, y[p], x[p]) - M[p]) * r[p];
                PixVec<P>::store(prob + n * C * hw + off + c * hw, o);
            }
        }
    }
}

// ---- in-training visualisation maps (utilities/utils.py:76-133, next-row component SURVEY.md 8f-4) -------------------------
// predictions = argmax_c(main + aux/2) (first maximal index, as torch.max), kld = PixelwiseKLD(main, aux), and the maximum of
// kld over the whole batch as an order-preserving key (float_to_key) folded with atomicMax -- what the reference gets from
// torch.max(kld).item() after three library passes and a host sync.
template <int P>
__global__ void __launch_bounds__(256) prediction_maps_kernel(const float* __restrict__ main_l, const float* __restrict__ aux_l,
                                                              int64_t n_img, int C, int64_t hw, long long* __restrict__ labels,
                                                              float* __restrict__ kld, unsigned int* __restrict__ kld_max_key) {
    const int64_t gpi = hw / P, n_groups = n_img * gpi;
    unsigned int best_key = 0;
    for (int64_t g = blockIdx.x * 256ll + threadIdx.x; g < n_groups; g += (int64_t)gridDim.x * 256) {
        const int64_t n = g / gpi, off = (g - n * gpi) * P;
        const float* pm = main_l + n * C * hw + off;
        const float* pa = aux_l ? aux_l + n * C * hw + off : nullptr;
        float zmax[P];
        int amax[P];
#pragma unroll
        for (int p = 0; p < P; ++p) { zmax[p] = -INFINITY; amax[p] = 0; }
        for (int c = 0; c < C; ++c) {
            float x[P], y[P];
            PixVec<P>::load(pm + c * hw, x);
            if (pa) PixVec<P>::load(pa + c * hw, y);
#pragma unroll
            for (int p = 0; p < P; ++p) {
                const float z = pa ? fmaf(0.5f, y[p], x[p]) : x[p];
                if (z > zmax[p] || c == 0) { zmax[p] = z; amax[p] = c; }      // strict >: first maximal index
            }
        }
#pragma unroll
        for (int p = 0; p < P; ++p) labels[n * hw + off + p] = amax[p];
        if (kld && pa) {
            KldStats<P> ks;
            kld_stats<P>(pm, pa, C, hw, ks);
            PixVec<P>::store(kld + n * hw + off, ks.D);
#pragma unroll
            for (int p = 0; p < P; ++p) best_key = max(best_key, float_to_key(ks.D[p]));
        }
    }
    if (kld_max_key) {
        best_key = __reduce_max_sync(0xffffffffu, best_key);
        if ((threadIdx.x & 31) == 0 && best_key) atomicMax(kld_max_key, best_key);
    }
}

// heat = -kld / max(kld) + 1 with IEEE fp32 division, exactly the reference's expression (utilities/utils.py:92, 103)
__global__ void __launch_bounds__(256) kld_heatmap_kernel(const float* __restrict__ kld, int64_t count,
                                                          const unsigned int* __restrict__ kld_max_key, float* __restrict__ heat) {
    const float mx = key_to_float(*kld_max_key);
    for (int64_t i = blockIdx.x * 256ll + threadIdx.x; i < count; i += (int64_t)gridDim.x * 256)
        heat[i] = __fadd_rn(__fdiv_rn(-kld[i], mx), 1.0f);
}

struct ColorTable { unsigned char rgb[256][3]; int n; };

// LongTensorToRGBPIL (utilities/utils.py:188-237) for a whole batch: labels (n, hw) int64 -> rgb (n, 3, hw) u8; labels outside
// the table give black (the reference leaves those bytes uninitialised)
__global__ void __launch_bounds__(256) label_colors_kernel(const long long* __restrict__ labels, int64_t n_img, int64_t hw,
                                                           const __grid_constant__ ColorTable tab, uint8_t* __restrict__ rgb) {
    for (int64_t i = blockIdx.x * 256ll + threadIdx.x; i < n_img * hw; i += (int64_t)gridDim.x * 256) {
        const int64_t n = i / hw, px = i - n * hw;
        const long long l = labels[i];
        const bool ok = l >= 0 && l < tab.n;
#pragma unroll
        for (int ch = 0; ch < 3; ++ch) rgb[(n * 3 + ch) * hw + px] = ok ? tab.rgb[l][ch] : 0;
    }
}

// PixelwiseKLD backward: g1_c = g p1_c (log p1_c - log p2_c - D), g2_c = g (p2_c - p1_c)
template <int P>
__global__ void __launch_bounds__(256) kld_bwd_kernel(const float* __restrict__ d1, const float* __restrict__ d2, const float* __restrict__ gk,
                                                      int64_t n_img, int C, int64_t hw, float* __restrict__ g1, float* __restrict__ g2) {
    const int64_t gpi = hw / P, n_groups = n_img * gpi;
    for (int64_t g = blockIdx.x * 256ll + threadIdx.x; g < n_groups; g += (int64_t)gridDim.x * 256) {
        const int64_t n = g / gpi, off = (g - n * gpi) * P;
        const int64_t base = n * C * hw + off;
        KldStats<P> ks;
        kld_stats<P>(d1 + base, d2 + base, C, hw, ks);
        float up[P], l1[P], l2[P], r1[P], r2[P];
        PixVec<P>::load(gk + n * hw + off, up);
#pragma unroll
        for (int p = 0; p < P; ++p) { l1[p] = logf(ks.S1[p]); l2[p] = logf(ks.S2[p]); r1[p] = 1.0f / ks.S1[p]; r2[p] = 1.0f / ks.S2[p]; }
        for (int c = 0; c < C; ++c) {
            float x[P], y[P], o1[P], o2[P];
            PixVec<P>::load(d1 + base + c * hw, x);
            PixVec<P>::load(d2 + base + c * hw, y);
#pragma unroll
            for (int p = 0; p < P; ++p) {
                const float t1 = x[p] - ks.M1[p], t2 = y[p] - ks.M2[p];
                const float p1 = exp_neg(t1) * r1[p], p2 = exp_neg(t2) * r2[p];
                o1[p] = up[p] * p1 * ((t1 - l1[p]) - (t2 - l2[p]) - ks.D[p]);
                o2[p] = up[p] * (p2 - p1);
            }
            PixVec<P>::store(g1 + base + c * hw, o1);
            PixVec<P>::store(g2 + base + c * hw, o2);
        }
    }
}

// UncertaintyWeightedSegmentationLoss forward / backward (loss_fns/segmentation_loss.py:155-175)
template <int P, bool BWD>
__global__ void __launch_bounds__(kLossThreads) uw_loss_kernel(const float* __restrict__ pred, const int64_t* __restrict__ target,
                                                               const float* __restrict__ u, const float* __restrict__ cw,
                                                               const float* __restrict__ grad_loss, int64_t n_img, int C, int64_t hw,
                                                               double inv_n, float* __restrict__ loss, float* __restrict__ d_pred,
                                                               float* __restrict__ d_u, LossWorkspace* ws) {
    const int64_t gpi = hw / P, n_groups = n_img * gpi;
    const float inv_nf = (float)inv_n;
    const float up = BWD ? grad_loss[0] : 0.f;
    double acc = 0;
    for (int64_t g = blockIdx.x * (int64_t)kLossThreads + threadIdx.x; g < n_groups; g += (int64_t)gridDim.x * kLossThreads) {
        const int64_t n = g / gpi, off = (g - n * gpi) * P;
        const float* pp = pred + n * C * hw + off;
        float M[P], S[P], uu[P], wt[P], l[P], eu[P], r[P];
        int ti[P];
        stats1<P>(pp, C, hw, M, S);
        PixVec<P>::load(u + n * hw + off, uu);
#pragma unroll
        for (int p = 0; p < P; ++p) {
            const long long t = target[n * hw + off + p];
            const bool valid = t >= 0 && t < C;
            ti[p] = valid ? (int)t : -1;
            wt[p] = valid ? __ldg(cw + t) : 0.f;
            const float xt = valid ? __ldg(pp + t * hw + p) : M[p];
            eu[p] = expf(-uu[p]);
            l[p] = wt[p] * (logf(S[p]) - (xt - M[p])) * eu[p];
            r[p] = 1.0f / S[p];
            acc += (double)l[p];
        }
        if (BWD) {
            for (int c = 0; c < C; ++c) {
                float x[P], o[P];
                PixVec<P>::load(pp + c * hw, x);
#pragma unroll
                for (int p = 0; p < P; ++p)
                    o[p] = up * inv_nf * eu[p] * wt[p] * (exp_neg(x[p] - M[p]) * r[p] - (ti[p] == c ? 1.0f : 0.0f));
                PixVec<P>::store(d_pred + n * C * hw + off + c * hw, o);
            }
            if (d_u) {
                float o[P];
#pragma unroll
                for (int p = 0; p < P; ++p) o[p] = -up * inv_nf * l[p];
                PixVec<P>::store(d_u + n * hw + off, o);
            }
        }
    }
    if (!BWD) finish_loss<1>(acc, 0.0, ws, inv_n, 1.0f, loss);
}

// ---- small class counts (C <= 8): logits live in registers, HBM and L2 see every value exactly once ----------------------
// PixelwiseKLD forward (BWD = false: writes D) / backward (BWD = true: reads the upstream gradient, writes g1, g2).
template <int P, int C, bool BWD>
__global__ void __launch_bounds__(256) kld_small_kernel(const float* __restrict__ d1, const float* __restrict__ d2, const float* __restrict__ up,
                                                        int64_t n_img, int64_t hw, float* __restrict__ kld, float* __restrict__ g1,
                                                        float* __restrict__ g2) {
    const int64_t gpi = hw / P, n_groups = n_img * gpi;
    for (int64_t g = blockIdx.x * 256ll + threadIdx.x; g < n_groups; g += (int64_t)gridDim.x * 256) {
        const int64_t n = g / gpi, off = (g - n * gpi) * P;
        const int64_t base = n * C * hw + off;
        float x[C][P], y[C][P], u[P];
#pragma unroll
        for (int c = 0; c < C; ++c) PixVec<P>::load(d1 + base + c * hw, x[c]);
#pragma unroll
        for (int c = 0; c < C; ++c) PixVec<P>::load(d2 + base + c * hw, y[c]);
        if (BWD) PixVec<P>::load(up + n * hw + off, u);
        float D[P];
#pragma unroll
        for (int p = 0; p < P; ++p) {
            float M1 = -INFINITY, M2 = -INFINITY;
#pragma unroll
            for (int c = 0; c < C; ++c) { M1 = fmaxf(M1, x[c][p]); M2 = fmaxf(M2, y[c][p]); }
            float e1[C], e2[C], S1 = 0.f, S2 = 0.f;
#pragma unroll
            for (int c = 0; c < C; ++c) {
                e1[c] = exp_neg(x[c][p] - M1); e2[c] = exp_neg(y[c][p] - M2);
                S1 += e1[c]; S2 += e2[c];
            }
            const float r1 = rcp_fast(S1), r2 = rcp_fast(S2), lr = log_fast(S1 * r2);     // log S1 - log S2
            float dl[C], d = 0.f;
#pragma unroll
            for (int c = 0; c < C; ++c) {
                dl[c] = ((x[c][p] - M1) - (y[c][p] - M2)) - lr;                             // log p1 - log p2
                d = fmaf(e1[c] * r1, dl[c], d);
            }
            D[p] = d;
            if (BWD) {
#pragma unroll
                for (int c = 0; c < C; ++c) {
                    const float p1 = e1[c] * r1, p2 = e2[c] * r2;
                    x[c][p] = u[p] * p1 * (dl[c] - d);
                    y[c][p] = u[p] * (p2 - p1);
                }
            }
        }
        if (BWD) {
#pragma unroll
            for (int c = 0; c < C; ++c) PixVec<P>::store(g1 + base + c * hw, x[c]);
#pragma unroll
            for (int c = 0; c < C; ++c) PixVec<P>::store(g2 + base + c * hw, y[c]);
        } else {
            PixVec<P>::store(kld + n * hw + off, D);
        }
    }
}

// UncertaintyWeightedSegmentationLoss forward / backward with the logits in registers.
template <int P, int C, bool BWD>
__global__ void __launch_bounds__(kLossThreads) uw_small_kernel(const float* __restrict__ pred, const int64_t* __restrict__ target,
                                                                const float* __restrict__ u, const float* __restrict__ cw,
                                                                const float* __restrict__ grad_loss, int64_t n_img, int64_t hw,
                                                                double inv_n, float* __restrict__ loss, float* __restrict__ d_pred,
                                                                float* __restrict__ d_u, LossWorkspace* ws) {
    __shared__ float s_w[C];
    if (threadIdx.x < C) s_w[threadIdx.x] = cw[threadIdx.x];
    __syncthreads();
    const int64_t gpi = hw / P, n_groups = n_img * gpi;
    const float inv_nf = (float)inv_n;
    const float upg = BWD ? grad_loss[0] * inv_nf : 0.f;
    double acc = 0;
    for (int64_t g = blockIdx.x * (int64_t)kLossThreads + threadIdx.x; g < n_groups; g += (int64_t)gridDim.x * kLossThreads) {
        const int64_t n = g / gpi, off = (g - n * gpi) * P;
        const int64_t base = n * C * hw + off;
        float x[C][P], uu[P], du[P];
#pragma unroll
        for (int c = 0; c < C; ++c) PixVec<P>::load(pred + base + c * hw, x[c]);
        PixVec<P>::load(u + n * hw + off, uu);
        float lsum = 0.f;
#pragma unroll
        for (int p = 0; p < P; ++p) {
            const long long t = __ldcs(target + n * hw + off + p);
            const bool valid = t >= 0 && t < C;
            const int ti = valid ? (int)t : -1;
            float M = -INFINITY;
#pragma unroll
            for (int c = 0; c < C; ++c) M = fmaxf(M, x[c][p]);
            float e[C], S = 0.f, wt = 0.f, xt = M;
#pragma unroll
            for (int c = 0; c < C; ++c) {
                e[c] = exp_neg(x[c][p] - M);
                S += e[c];
                wt = (ti == c) ? s_w[c] : wt;
                xt = (ti == c) ? x[c][p] : xt;
            }
            const float eu = exp_neg(-uu[p]);
            const float l = wt * (log_fast(S) - (xt - M)) * eu;
            lsum += l;
            if (BWD) {
                const float r = rcp_fast(S), coef = upg * eu * wt;
#pragma unroll
                for (int c = 0; c < C; ++c) x[c][p] = coef * (e[c] * r - (ti == c ? 1.0f : 0.0f));
                du[p] = -upg * l;
            }
        }
        acc += (double)lsum;
        if (BWD) {
#pragma unroll
            for (int c = 0; c < C; ++c) PixVec<P>::store(d_pred + base + c * hw, x[c]);
            if (d_u) PixVec<P>::store(d_u + n * hw + off, du);
        }
    }
    if (!BWD) finish_loss<1>(acc, 0.0, ws, inv_n, 1.0f, loss);
}

__global__ void __launch_bounds__(256) scale_inplace_kernel(float* __restrict__ x, int64_t count, const float* __restrict__ scale) {
    const float s = scale[0];
    if (s == 1.0f) return;
    for (int64_t i = blockIdx.x * 256ll + threadIdx.x; i < count; i += (int64_t)gridDim.x * 256) x[i] *= s;
}

static int64_t persistent_grid(int64_t n_groups, int threads, int per_sm, int64_t cap) {
    int64_t blocks = (n_groups + threads - 1) / threads;
    const int64_t lim = (int64_t)kNumSMs * per_sm < cap ? (int64_t)kNumSMs * per_sm : cap;
    return blocks < 1 ? 1 : (blocks < lim ? blocks : lim);
}

// Pixels per thread when rows are 16-byte aligned, picked on B200 (profiles/r01_loss_variants.txt): the backward keeps
// 2*K*P gradient registers live, so it wants the narrower P=2 (77% of the measured HBM peak vs 68% at P=4); the
// forward-only kernel is best at P=4 (76% vs 63%).
// Persistent grid of exactly the CTAs that are resident at once (occupancy query), so no second wave.
template <typename Kern>
static int64_t resident_grid(Kern kern, int64_t n_groups) {
    int dev = 0, sms = kNumSMs, per_sm = 2;
    if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, kLossThreads, 0) != cudaSuccess || per_sm < 1) {
        cudaGetLastError();
        per_sm = 2;
    }
    const int64_t blocks = (n_groups + kLossThreads - 1) / kLossThreads;
    const int64_t cap = std::min<int64_t>((int64_t)sms * per_sm, kMaxLossBlocks);
    return blocks < 1 ? 1 : (blocks < cap ? blocks : cap);
}

// Pixels per thread of the vector path for fp16 / bf16 logits (profiles/r05_loss_half_variants.txt).  Needs hw % P == 0 and
// every plane 2P-byte aligned; otherwise P = 1.
constexpr int kHalfFwdP = 4;
constexpr int kHalfBwdP = 2;
template <typename LT> constexpr int vec_pixels(bool bwd) {
    return sizeof(LT) == 4 ? (bwd ? MSPL_UWCE_BWD_P : 4) : (bwd ? kHalfBwdP : kHalfFwdP);
}

template <int K, typename TT, bool IOU, typename LT>
static int launch_uw_ce(bool vec, bool bwd, const LT* m, const LT* a, const TT* t, const float* cw, int64_t n, int64_t hw,
                        float alpha, double inv_n, float gs, const float* gs_dev, float* out3, LT* dm, LT* da, LossWorkspace* ws,
                        unsigned long long* iou, cudaStream_t st) {
    constexpr int PF = vec_pixels<LT>(false), PB = vec_pixels<LT>(true);
    const int pv = vec ? (bwd ? PB : PF) : 1;
    const int64_t n_groups = n * (hw / pv);
#define MSPL_UWCE(PP, BB)                                                                                                  \
    {                                                                                                                      \
        if constexpr (sizeof(LT) == 4) {                                                                                   \
            auto kern = uw_ce_fused_kernel<PP, K, BB, TT, IOU>;                                                            \
            kern<<<(unsigned)resident_grid(kern, n_groups), kLossThreads, 0, st>>>(m, a, t, cw, n, hw, alpha, inv_n, gs, out3, dm, da, \
                                                                                   ws, iou);                                \
        } else {                                                                                                           \
            auto kern = uw_ce_fused_half_kernel<PP, K, BB, TT, IOU, LT>;                                                   \
            kern<<<(unsigned)resident_grid(kern, n_groups), kLossThreads, 0, st>>>(m, a, t, cw, n, hw, alpha, inv_n, gs, out3, dm, da, \
                                                                                   ws, iou, gs_dev);                        \
        }                                                                                                                  \
    }
    if (vec && !bwd) MSPL_UWCE(PF, false)
    else if (vec) MSPL_UWCE(PB, true)
    else if (bwd) MSPL_UWCE(1, true)
    else MSPL_UWCE(1, false)
#undef MSPL_UWCE
    return launch_status();
}

}  // namespace mspl

using namespace mspl;

extern "C" size_t mspl_uw_ce_workspace_bytes(void) { return sizeof(LossWorkspace); }

template <typename TT, typename LT>
static int uw_ce_entry(const LT* main_logits, const LT* aux_logits, const TT* target, const float* class_weights,
                       int64_t num_images, int num_classes, int64_t pixels_per_image, float alpha, double norm_pixels,
                       float grad_scale, const float* grad_scale_dev, float* out3, LT* d_main, LT* d_aux, void* workspace,
                       size_t workspace_bytes, unsigned long long* iou_counts, void* stream) {
    if (!main_logits || !aux_logits || !target || !class_weights || !out3 || !workspace) return MSPL_ERR_BAD_ARG;
    if (!aligned_to(iou_counts, 8)) return MSPL_ERR_ALIGN;
    if ((d_main == nullptr) != (d_aux == nullptr)) return MSPL_ERR_BAD_ARG;
    if (num_images < 1 || pixels_per_image < 1 || num_classes < 1 || !(norm_pixels > 0)) return MSPL_ERR_BAD_ARG;
    if (workspace_bytes < sizeof(LossWorkspace)) return MSPL_ERR_WORKSPACE;
    if (num_classes > MSPL_MAX_CLASSES) return MSPL_ERR_UNSUPPORTED;
    if (!aligned_to(main_logits, sizeof(LT)) || !aligned_to(aux_logits, sizeof(LT)) || !aligned_to(d_main, sizeof(LT)) ||
        !aligned_to(d_aux, sizeof(LT)) || !aligned_to(target, sizeof(TT)) || !aligned_to(workspace, 8) ||
        !aligned_to(grad_scale_dev, 4))
        return MSPL_ERR_ALIGN;
    const bool bwd = d_main != nullptr;
    bool vec;
    if (sizeof(LT) == 4) {
        // widest group of pixels per thread: rows of logits 16-byte aligned, and the group's targets loadable as one vector
        // (two 16-byte loads of int64, one 4-byte load of uint8; the backward takes half a group)
        vec = pick_vec(pixels_per_image, {main_logits, aux_logits, d_main, d_aux}) == 4 && aligned_to(target, sizeof(TT) == 8 ? 16 : 4);
    } else {
        // P 2-byte pixels per thread: P-pixel rows, every plane 2P-byte aligned, the targets as 16-byte (int64) or P-byte loads
        const int P = vec_pixels<LT>(bwd);
        vec = pixels_per_image % P == 0 && aligned_to(target, sizeof(TT) == 8 ? 16 : P);
        for (const void* q : {(const void*)main_logits, (const void*)aux_logits, (const void*)d_main, (const void*)d_aux})
            vec = vec && aligned_to(q, 2 * P);
    }
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    LossWorkspace* ws = static_cast<LossWorkspace*>(workspace);
    const double inv_n = 1.0 / norm_pixels;
#define MSPL_CASE(KK)                                                                                                            \
    case KK:                                                                                                                     \
        return iou_counts ? launch_uw_ce<KK, TT, true>(vec, bwd, main_logits, aux_logits, target, class_weights, num_images,      \
                                                       pixels_per_image, alpha, inv_n, grad_scale, grad_scale_dev, out3, d_main,  \
                                                       d_aux, ws, iou_counts, st)                                                 \
                          : launch_uw_ce<KK, TT, false>(vec, bwd, main_logits, aux_logits, target, class_weights, num_images,     \
                                                        pixels_per_image, alpha, inv_n, grad_scale, grad_scale_dev, out3, d_main, \
                                                        d_aux, ws, nullptr, st)
    switch (num_classes) {
        MSPL_CASE(1); MSPL_CASE(2); MSPL_CASE(3); MSPL_CASE(4); MSPL_CASE(5); MSPL_CASE(6); MSPL_CASE(7); MSPL_CASE(8);
    }
#undef MSPL_CASE
    return MSPL_ERR_UNSUPPORTED;
}

extern "C" int mspl_uw_ce_fwd_bwd(const float* main_logits, const float* aux_logits, const int64_t* target, const float* class_weights,
                                  int64_t num_images, int num_classes, int64_t pixels_per_image, float alpha, double norm_pixels,
                                  float grad_scale, float* out3, float* d_main, float* d_aux, void* workspace, size_t workspace_bytes,
                                  void* stream) {
    return uw_ce_entry<int64_t>(main_logits, aux_logits, target, class_weights, num_images, num_classes, pixels_per_image, alpha,
                                norm_pixels, grad_scale, nullptr, out3, d_main, d_aux, workspace, workspace_bytes, nullptr, stream);
}

extern "C" int mspl_uw_ce_fwd_bwd_u8(const float* main_logits, const float* aux_logits, const uint8_t* target, const float* class_weights,
                                     int64_t num_images, int num_classes, int64_t pixels_per_image, float alpha, double norm_pixels,
                                     float grad_scale, float* out3, float* d_main, float* d_aux, void* workspace,
                                     size_t workspace_bytes, void* stream) {
    return uw_ce_entry<uint8_t>(main_logits, aux_logits, target, class_weights, num_images, num_classes, pixels_per_image, alpha,
                                norm_pixels, grad_scale, nullptr, out3, d_main, d_aux, workspace, workspace_bytes, nullptr, stream);
}

extern "C" int mspl_uw_ce_step(const float* main_logits, const float* aux_logits, const void* target, int target_is_u8,
                               const float* class_weights, int64_t num_images, int num_classes, int64_t pixels_per_image, float alpha,
                               double norm_pixels, float grad_scale, float* out3, float* d_main, float* d_aux,
                               unsigned long long* iou_counts, void* workspace, size_t workspace_bytes, void* stream) {
    if (target_is_u8)
        return uw_ce_entry<uint8_t>(main_logits, aux_logits, static_cast<const uint8_t*>(target), class_weights, num_images,
                                    num_classes, pixels_per_image, alpha, norm_pixels, grad_scale, nullptr, out3, d_main, d_aux,
                                    workspace, workspace_bytes, iou_counts, stream);
    return uw_ce_entry<int64_t>(main_logits, aux_logits, static_cast<const int64_t*>(target), class_weights, num_images, num_classes,
                                pixels_per_image, alpha, norm_pixels, grad_scale, nullptr, out3, d_main, d_aux, workspace,
                                workspace_bytes, iou_counts, stream);
}

extern "C" int mspl_uw_ce_step_half(const void* main_logits, const void* aux_logits, int logit_dtype, const void* target,
                                    int target_is_u8, const float* class_weights, int64_t num_images, int num_classes,
                                    int64_t pixels_per_image, float alpha, double norm_pixels, float grad_scale,
                                    const float* grad_scale_dev, float* out3, void* d_main, void* d_aux,
                                    unsigned long long* iou_counts, void* workspace, size_t workspace_bytes, void* stream) {
    auto run = [&](auto lt) {
        using LT = decltype(lt);
        const LT *m = static_cast<const LT*>(main_logits), *a = static_cast<const LT*>(aux_logits);
        LT *dm = static_cast<LT*>(d_main), *da = static_cast<LT*>(d_aux);
        if (target_is_u8)
            return uw_ce_entry<uint8_t, LT>(m, a, static_cast<const uint8_t*>(target), class_weights, num_images, num_classes,
                                            pixels_per_image, alpha, norm_pixels, grad_scale, grad_scale_dev, out3, dm, da,
                                            workspace, workspace_bytes, iou_counts, stream);
        return uw_ce_entry<int64_t, LT>(m, a, static_cast<const int64_t*>(target), class_weights, num_images, num_classes,
                                        pixels_per_image, alpha, norm_pixels, grad_scale, grad_scale_dev, out3, dm, da, workspace,
                                        workspace_bytes, iou_counts, stream);
    };
    if (logit_dtype == MSPL_DTYPE_F16) return run(__half());
    if (logit_dtype == MSPL_DTYPE_BF16) return run(__nv_bfloat16());
    return MSPL_ERR_BAD_ARG;
}

template <int K, typename TT>
static int launch_uw_ce_lowres(bool bwd, const float* m, const float* a, const TT* t, const float* cw, int64_t n, LowresGeom g,
                               float alpha, double inv_n, float gs, float* out3, float* dm, float* da, LossWorkspace* ws, cudaStream_t st) {
    int dev = 0, sms = kNumSMs, max_smem = 227 * 1024;
    if (cudaGetDevice(&dev) == cudaSuccess) {
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        cudaDeviceGetAttribute(&max_smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
    }
    size_t smem = 0;
    for (int tr = 8; tr >= 1; tr >>= 1) {          // tallest tile whose gradients fit in shared memory
        g.TR = tr;
        g.nrm = std::min(g.hm, (int)(g.rhm * (float)(tr - 1)) + 3);
        g.nra = std::min(g.ha, (int)(g.rha * (float)(tr - 1)) + 3);
        smem = lowres_smem_bytes(g, K, bwd);
        if (smem <= (size_t)max_smem) break;
        if (tr == 1) return MSPL_ERR_UNSUPPORTED;   // image too wide for one row of gradients in shared memory
    }
    g.tiles_per_img = (g.H + g.TR - 1) / g.TR;
    const int64_t n_tiles = n * g.tiles_per_img;
    auto launch = [&](auto kern) {
        if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) {
            cudaGetLastError();
            return (int)MSPL_ERR_CUDA;
        }
        int per_sm = 1;         // persistent grid of the CTAs that are resident at once (1 with a tile of gradients, more without)
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, kLowresThreads, smem) != cudaSuccess || per_sm < 1) {
            cudaGetLastError();
            per_sm = 1;
        }
        const int64_t grid = std::min<int64_t>(n_tiles, std::min<int64_t>((int64_t)sms * per_sm, kMaxLossBlocks));
        kern<<<(unsigned)grid, kLowresThreads, smem, st>>>(m, a, t, cw, n, g, alpha, inv_n, gs, out3, dm, da, ws);
        return launch_status();
    };
    return bwd ? launch(uw_ce_lowres_kernel<K, true, TT>) : launch(uw_ce_lowres_kernel<K, false, TT>);
}

template <typename TT>
static int uw_ce_lowres_entry(const float* main_lowres, const float* aux_lowres, const TT* target, const float* class_weights,
                              int64_t num_images, int num_classes, int main_h, int main_w, int aux_h, int aux_w, int out_h, int out_w,
                              float alpha, double norm_pixels, float grad_scale, float* out3, float* d_main_lowres,
                              float* d_aux_lowres, void* workspace, size_t workspace_bytes, void* stream) {
    if (!main_lowres || !aux_lowres || !target || !class_weights || !out3 || !workspace) return MSPL_ERR_BAD_ARG;
    if ((d_main_lowres == nullptr) != (d_aux_lowres == nullptr)) return MSPL_ERR_BAD_ARG;
    if (num_images < 1 || num_classes < 1 || !(norm_pixels > 0)) return MSPL_ERR_BAD_ARG;
    if (main_h < 1 || main_w < 1 || aux_h < 1 || aux_w < 1 || out_h < 1 || out_w < 1) return MSPL_ERR_BAD_ARG;
    if (workspace_bytes < sizeof(LossWorkspace)) return MSPL_ERR_WORKSPACE;
    if (num_classes > MSPL_MAX_CLASSES) return MSPL_ERR_UNSUPPORTED;
    if (main_h > out_h || main_w > out_w || aux_h > out_h || aux_w > out_w) return MSPL_ERR_UNSUPPORTED;   // upsampling only
    if ((int64_t)out_h * out_w >= (1ll << 24)) return MSPL_ERR_UNSUPPORTED;
    if (!aligned_to(main_lowres, 4) || !aligned_to(aux_lowres, 4) || !aligned_to(target, sizeof(TT)) || !aligned_to(workspace, 8) ||
        !aligned_to(d_main_lowres, 4) || !aligned_to(d_aux_lowres, 4))
        return MSPL_ERR_ALIGN;
    const bool bwd = d_main_lowres != nullptr;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    LowresGeom g{};
    g.hm = main_h; g.wm = main_w; g.ha = aux_h; g.wa = aux_w; g.H = out_h; g.W = out_w;
    // ATen's area_pixel_compute_scale for align_corners=True, evaluated in fp32 like the CUDA upsample kernel does
    auto scale = [](int in, int out) { return out > 1 ? (float)(in - 1) / (float)(out - 1) : 0.f; };
    g.rhm = scale(main_h, out_h); g.rwm = scale(main_w, out_w); g.rha = scale(aux_h, out_h); g.rwa = scale(aux_w, out_w);
    g.inv_w = 1.0f / (float)out_w;
    if (bwd) {      // the tiles ADD their shares: start from zero (enqueued on the stream like the kernel itself)
        const size_t nm = (size_t)num_images * num_classes * main_h * main_w, na = (size_t)num_images * num_classes * aux_h * aux_w;
        if (cudaMemsetAsync(d_main_lowres, 0, nm * sizeof(float), st) != cudaSuccess ||
            cudaMemsetAsync(d_aux_lowres, 0, na * sizeof(float), st) != cudaSuccess) {
            cudaGetLastError();
            return MSPL_ERR_CUDA;
        }
    }
    LossWorkspace* ws = static_cast<LossWorkspace*>(workspace);
    const double inv_n = 1.0 / norm_pixels;
#define MSPL_CASE(KK) case KK: return launch_uw_ce_lowres<KK, TT>(bwd, main_lowres, aux_lowres, target, class_weights, num_images, g, alpha, inv_n, grad_scale, out3, d_main_lowres, d_aux_lowres, ws, st)
    switch (num_classes) {
        MSPL_CASE(1); MSPL_CASE(2); MSPL_CASE(3); MSPL_CASE(4); MSPL_CASE(5); MSPL_CASE(6); MSPL_CASE(7); MSPL_CASE(8);
    }
#undef MSPL_CASE
    return MSPL_ERR_UNSUPPORTED;
}

#define MSPL_LOWRES_ARGS                                                                                                          \
    main_lowres, aux_lowres, target, class_weights, num_images, num_classes, main_h, main_w, aux_h, aux_w, out_h, out_w, alpha,      \
        norm_pixels, grad_scale, out3, d_main_lowres, d_aux_lowres, workspace, workspace_bytes, stream

extern "C" int mspl_uw_ce_lowres_fwd_bwd(const float* main_lowres, const float* aux_lowres, const int64_t* target,
                                         const float* class_weights, int64_t num_images, int num_classes, int main_h, int main_w,
                                         int aux_h, int aux_w, int out_h, int out_w, float alpha, double norm_pixels, float grad_scale,
                                         float* out3, float* d_main_lowres, float* d_aux_lowres, void* workspace, size_t workspace_bytes,
                                         void* stream) {
    return uw_ce_lowres_entry<int64_t>(MSPL_LOWRES_ARGS);
}

extern "C" int mspl_uw_ce_lowres_fwd_bwd_u8(const float* main_lowres, const float* aux_lowres, const uint8_t* target,
                                            const float* class_weights, int64_t num_images, int num_classes, int main_h, int main_w,
                                            int aux_h, int aux_w, int out_h, int out_w, float alpha, double norm_pixels,
                                            float grad_scale, float* out3, float* d_main_lowres, float* d_aux_lowres, void* workspace,
                                            size_t workspace_bytes, void* stream) {
    return uw_ce_lowres_entry<uint8_t>(MSPL_LOWRES_ARGS);
}
#undef MSPL_LOWRES_ARGS

extern "C" int mspl_scale_inplace(float* x, int64_t count, const float* scale, void* stream) {
    if (!x || !scale || count < 0) return MSPL_ERR_BAD_ARG;
    if (count == 0) return MSPL_OK;
    const int64_t grid = persistent_grid(count, 256, 8, 1 << 20);
    scale_inplace_kernel<<<(unsigned)grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(x, count, scale);
    return launch_status();
}

static bool bad_planes(const void* a, const void* b, int64_t n, int c, int64_t hw) {
    return !a || !b || n < 0 || c < 1 || hw < 1;
}

extern "C" int mspl_softmax_kld(const float* main_logits, const float* aux_logits, int64_t n, int c, int64_t pixels_per_image,
                                float* prob, float* kld, void* stream) {
    if (bad_planes(main_logits, aux_logits, n, c, pixels_per_image) || (!prob && !kld)) return MSPL_ERR_BAD_ARG;
    if (n == 0) return MSPL_OK;
    const int P = pick_vec(pixels_per_image, {main_logits, aux_logits, prob, kld}) == 4 ? 4 : 1;
    const int64_t grid = persistent_grid(n * (pixels_per_image / P), 256, 8, 1 << 20);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (P == 4) softmax_kld_kernel<4><<<(unsigned)grid, 256, 0, st>>>(main_logits, aux_logits, n, c, pixels_per_image, prob, kld);
    else softmax_kld_kernel<1><<<(unsigned)grid, 256, 0, st>>>(main_logits, aux_logits, n, c, pixels_per_image, prob, kld);
    return launch_status();
}

#define MSPL_SMALL_C_SWITCH(c, STMT)            \
    switch (c) {                                \
        case 2: { constexpr int CC = 2; STMT; } break; \
        case 3: { constexpr int CC = 3; STMT; } break; \
        case 4: { constexpr int CC = 4; STMT; } break; \
        case 5: { constexpr int CC = 5; STMT; } break; \
        case 6: { constexpr int CC = 6; STMT; } break; \
        case 7: { constexpr int CC = 7; STMT; } break; \
        case 8: { constexpr int CC = 8; STMT; } break; \
        default: break;                         \
    }

extern "C" int mspl_prediction_maps(const float* main_logits, const float* aux_logits, int64_t n, int c, int64_t pixels_per_image,
                                    int64_t* labels, float* kld, unsigned int* kld_max_key, void* stream) {
    if (!main_logits || !labels || n < 0 || c < 1 || pixels_per_image < 1) return MSPL_ERR_BAD_ARG;
    if ((kld || kld_max_key) && !aux_logits) return MSPL_ERR_BAD_ARG;
    if (kld_max_key && !kld) return MSPL_ERR_BAD_ARG;
    if (!aligned_to(main_logits, 4) || !aligned_to(aux_logits, 4) || !aligned_to(labels, 8) || !aligned_to(kld, 4) ||
        !aligned_to(kld_max_key, 4))
        return MSPL_ERR_ALIGN;
    if (n == 0) return MSPL_OK;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const int P = pick_vec(pixels_per_image, {main_logits, aux_logits, kld}) == 4 ? 4 : 1;
    const int64_t grid = persistent_grid(n * (pixels_per_image / P), 256, 8, 1 << 20);
    if (P == 4)
        prediction_maps_kernel<4><<<(unsigned)grid, 256, 0, st>>>(main_logits, aux_logits, n, c, pixels_per_image,
                                                                  reinterpret_cast<long long*>(labels), kld, kld_max_key);
    else
        prediction_maps_kernel<1><<<(unsigned)grid, 256, 0, st>>>(main_logits, aux_logits, n, c, pixels_per_image,
                                                                  reinterpret_cast<long long*>(labels), kld, kld_max_key);
    return launch_status();
}

extern "C" int mspl_kld_heatmap(const float* kld, int64_t count, const unsigned int* kld_max_key, float* heat, void* stream) {
    if (!kld || !kld_max_key || !heat || count < 0) return MSPL_ERR_BAD_ARG;
    if (!aligned_to(kld, 4) || !aligned_to(heat, 4) || !aligned_to(kld_max_key, 4)) return MSPL_ERR_ALIGN;
    if (count == 0) return MSPL_OK;
    kld_heatmap_kernel<<<(unsigned)persistent_grid(count, 256, 8, 1 << 20), 256, 0, static_cast<cudaStream_t>(stream)>>>(
        kld, count, kld_max_key, heat);
    return launch_status();
}

extern "C" int mspl_label_colors(const int64_t* labels, int64_t n, int64_t pixels_per_image, const uint8_t* colors_rgb, int num_colors,
                                 uint8_t* rgb, void* stream) {
    if (!labels || !colors_rgb || !rgb || n < 0 || pixels_per_image < 1 || num_colors < 0 || num_colors > 256) return MSPL_ERR_BAD_ARG;
    if (!aligned_to(labels, 8)) return MSPL_ERR_ALIGN;
    if (n == 0) return MSPL_OK;
    ColorTable tab;
    memset(&tab, 0, sizeof(tab));
    tab.n = num_colors;
    for (int i = 0; i < num_colors; ++i)
        for (int ch = 0; ch < 3; ++ch) tab.rgb[i][ch] = colors_rgb[3 * i + ch];
    label_colors_kernel<<<(unsigned)persistent_grid(n * pixels_per_image, 256, 8, 1 << 20), 256, 0, static_cast<cudaStream_t>(stream)>>>(
        reinterpret_cast<const long long*>(labels), n, pixels_per_image, tab, rgb);
    return launch_status();
}

extern "C" int mspl_kld_fwd(const float* dist1, const float* dist2, int64_t n, int c, int64_t pixels_per_image, float* kld, void* stream) {
    if (!kld) return MSPL_ERR_BAD_ARG;
    if (c >= 2 && c <= 8 && dist1 && dist2 && n > 0 && pixels_per_image > 0 &&
        pick_vec(pixels_per_image, {dist1, dist2, kld}) == 4) {
        const int64_t grid = persistent_grid(n * (pixels_per_image / 4), 256, 4, 1 << 20);
        cudaStream_t st = static_cast<cudaStream_t>(stream);
        MSPL_SMALL_C_SWITCH(c, (kld_small_kernel<4, CC, false><<<(unsigned)grid, 256, 0, st>>>(dist1, dist2, nullptr, n, pixels_per_image, kld, nullptr, nullptr)));
        return launch_status();
    }
    return mspl_softmax_kld(dist1, dist2, n, c, pixels_per_image, nullptr, kld, stream);
}

extern "C" int mspl_kld_bwd(const float* dist1, const float* dist2, const float* grad_kld, int64_t n, int c, int64_t pixels_per_image,
                            float* grad1, float* grad2, void* stream) {
    if (bad_planes(dist1, dist2, n, c, pixels_per_image) || !grad_kld || !grad1 || !grad2) return MSPL_ERR_BAD_ARG;
    if (n == 0) return MSPL_OK;
    if (c >= 2 && c <= 8 && pick_vec(pixels_per_image, {dist1, dist2, grad_kld, grad1, grad2}) == 4) {
        const int64_t grid = persistent_grid(n * (pixels_per_image / 2), 256, 4, 1 << 20);
        cudaStream_t st = static_cast<cudaStream_t>(stream);
        MSPL_SMALL_C_SWITCH(c, (kld_small_kernel<2, CC, true><<<(unsigned)grid, 256, 0, st>>>(dist1, dist2, grad_kld, n, pixels_per_image, nullptr, grad1, grad2)));
        return launch_status();
    }
    const int P = pick_vec(pixels_per_image, {dist1, dist2, grad_kld, grad1, grad2}) == 4 ? 4 : 1;
    const int64_t grid = persistent_grid(n * (pixels_per_image / P), 256, 8, 1 << 20);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (P == 4) kld_bwd_kernel<4><<<(unsigned)grid, 256, 0, st>>>(dist1, dist2, grad_kld, n, c, pixels_per_image, grad1, grad2);
    else kld_bwd_kernel<1><<<(unsigned)grid, 256, 0, st>>>(dist1, dist2, grad_kld, n, c, pixels_per_image, grad1, grad2);
    return launch_status();
}

extern "C" int mspl_uw_loss_fwd(const float* pred, const int64_t* target, const float* u_weight, const float* class_weights, int64_t n,
                                int num_classes, int64_t pixels_per_image, double norm_pixels, float* loss, void* workspace,
                                size_t workspace_bytes, void* stream) {
    if (!pred || !target || !u_weight || !class_weights || !loss || !workspace) return MSPL_ERR_BAD_ARG;
    if (n < 1 || num_classes < 1 || pixels_per_image < 1 || !(norm_pixels > 0)) return MSPL_ERR_BAD_ARG;
    if (workspace_bytes < sizeof(LossWorkspace)) return MSPL_ERR_WORKSPACE;
    const int P = pick_vec(pixels_per_image, {pred, u_weight}) == 4 ? 4 : 1;
    const int64_t grid = persistent_grid(n * (pixels_per_image / P), kLossThreads, 4, kMaxLossBlocks);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    LossWorkspace* ws = static_cast<LossWorkspace*>(workspace);
    if (P == 4 && num_classes >= 2 && num_classes <= 8) {
        MSPL_SMALL_C_SWITCH(num_classes, (uw_small_kernel<4, CC, false><<<(unsigned)grid, kLossThreads, 0, st>>>(pred, target, u_weight, class_weights, nullptr, n, pixels_per_image, 1.0 / norm_pixels, loss, nullptr, nullptr, ws)));
        return launch_status();
    }
    if (P == 4) uw_loss_kernel<4, false><<<(unsigned)grid, kLossThreads, 0, st>>>(pred, target, u_weight, class_weights, nullptr, n, num_classes, pixels_per_image, 1.0 / norm_pixels, loss, nullptr, nullptr, ws);
    else uw_loss_kernel<1, false><<<(unsigned)grid, kLossThreads, 0, st>>>(pred, target, u_weight, class_weights, nullptr, n, num_classes, pixels_per_image, 1.0 / norm_pixels, loss, nullptr, nullptr, ws);
    return launch_status();
}

extern "C" int mspl_uw_loss_bwd(const float* pred, const int64_t* target, const float* u_weight, const float* class_weights,
                                const float* grad_loss, int64_t n, int num_classes, int64_t pixels_per_image, double norm_pixels,
                                float* d_pred, float* d_u, void* stream) {
    if (!pred || !target || !u_weight || !class_weights || !grad_loss || !d_pred) return MSPL_ERR_BAD_ARG;
    if (n < 1 || num_classes < 1 || pixels_per_image < 1 || !(norm_pixels > 0)) return MSPL_ERR_BAD_ARG;
    const int P = pick_vec(pixels_per_image, {pred, u_weight, d_pred, d_u}) == 4 ? 4 : 1;
    const int64_t grid = persistent_grid(n * (pixels_per_image / P), kLossThreads, 4, 1 << 20);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (P == 4 && num_classes >= 2 && num_classes <= 8) {
        MSPL_SMALL_C_SWITCH(num_classes, (uw_small_kernel<4, CC, true><<<(unsigned)grid, kLossThreads, 0, st>>>(pred, target, u_weight, class_weights, grad_loss, n, pixels_per_image, 1.0 / norm_pixels, nullptr, d_pred, d_u, nullptr)));
        return launch_status();
    }
    if (P == 4) uw_loss_kernel<4, true><<<(unsigned)grid, kLossThreads, 0, st>>>(pred, target, u_weight, class_weights, grad_loss, n, num_classes, pixels_per_image, 1.0 / norm_pixels, nullptr, d_pred, d_u, nullptr);
    else uw_loss_kernel<1, true><<<(unsigned)grid, kLossThreads, 0, st>>>(pred, target, u_weight, class_weights, grad_loss, n, num_classes, pixels_per_image, 1.0 / norm_pixels, nullptr, d_pred, d_u, nullptr);
    return launch_status();
}
