// Host-side launch helpers for the K1 kernels (shared by libmspl_b200.so and tools/k1_sweep).
#pragma once
#include <algorithm>
#include <cstring>

#include "fuse_kernel.cuh"

namespace mspl {

struct DeviceInfo {
    int sms = kNumSMs;
    bool ok = false;
};

inline DeviceInfo device_info() {
    DeviceInfo d;
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return d;
    if (cudaDeviceGetAttribute(&d.sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) return d;
    d.ok = true;
    return d;
}

// 1 + the index of the listed shape (kSourceShapes) that an order built for chunks of `chunk` classes has, or 0.
inline uint32_t listed_shape(const ClassOrder& o, int C, int chunk) {
    if (chunk != kFuseChunk) return 0;
    for (int i = 0; i < kNumSourceShapes; ++i) {
        const SourceShape& sh = kSourceShapes[i];
        if (sh.C == C && sh.nchunk == (int)o.nchunk && memcmp(sh.seg, o.seg, (size_t)sh.nchunk) == 0) return (uint32_t)i + 1;
    }
    return 0;
}

// Class visiting order of every source for chunks of `chunk` classes (see ClassOrder in pixel_math.cuh): classes sorted by
// (target class, class index); per chunk a byte with bit j = slot j ends its target group (chunk <= 8).
// Needs prm.S, prm.C and prm.lut; returns false when a source has more chunks than ClassOrder::seg holds.
inline bool build_class_order(FuseParams& prm, int chunk) {
    if (chunk > 8) return false;
    for (int s = 0; s < prm.S; ++s) {
        ClassOrder& o = prm.order[s];
        memset(&o, 0, sizeof(o));
        const int C = prm.C[s];
        if ((C + chunk - 1) / chunk > kMaxChunksPerSource) return false;
        o.nchunk = (uint32_t)((C + chunk - 1) / chunk);
        int i = 0;
        for (int k = 0; k < MSPL_MAX_CLASSES; ++k)
            for (int c = 0; c < C; ++c)
                if (prm.lut[s][c] == k) {
                    o.row[i++] = (uint8_t)c;
                    o.present |= 1u << k;
                }
        if (i != C) return false;            // a table entry >= MSPL_MAX_CLASSES (callers validate entries < K)
        for (int k = 0; k < MSPL_MAX_CLASSES; ++k)
            if ((o.present >> k) & 1u) o.vote[o.ngroup++] = 1u << (4 * k);
        for (i = 0; i < C; ++i) {
            const int k = prm.lut[s][o.row[i]];
            const bool last = (i == C - 1) || prm.lut[s][o.row[i + 1]] != k;
            if (last) o.seg[i / chunk] |= (uint8_t)(1u << (i % chunk));
        }
        o.shape = listed_shape(o, C, chunk);
    }
    return true;
}

// Persistent grid: one wave of resident CTAs, each striding over the pixel tiles.
template <int THREADS, typename Kern>
int launch_fuse_direct(Kern kern, const FuseParams& prm, int KT, cudaStream_t stream) {
    const size_t smem = fuse_tally_smem_bytes(prm.K, KT, THREADS, 1);
    const DeviceInfo di = device_info();
    int per_sm = 0;
    if (!di.ok || cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess ||
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, THREADS, smem) != cudaSuccess || per_sm < 1) {
        cudaGetLastError();
        return MSPL_ERR_CUDA;
    }
    const int64_t n_groups = prm.n_img * prm.hw;
    const int64_t n_tiles = (n_groups + THREADS - 1) / THREADS;
    const int64_t cap = (int64_t)di.sms * per_sm;
    kern<<<(unsigned)(n_tiles < cap ? n_tiles : cap), THREADS, smem, stream>>>(prm);
    return launch_status();
}

// The staged kernels (TMA, K1-lowres): one CTA per SM (the shared-memory ring fills the SM), striding over the tiles of
// Cfg::kTilePix pixels; smem: the kernel's dynamic shared memory (TmaCfg::smem_bytes, lowres_plan).
template <typename Cfg, typename Kern>
int launch_fuse_ring(Kern kern, const FuseParams& prm, size_t smem, cudaStream_t stream) {
    const DeviceInfo di = device_info();
    if (!di.ok || smem > 227 * 1024 || cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) {
        cudaGetLastError();
        return MSPL_ERR_CUDA;
    }
    const int64_t n_tiles = prm.n_img * ((prm.hw + Cfg::kTilePix - 1) / Cfg::kTilePix);
    kern<<<(unsigned)(n_tiles < di.sms ? n_tiles : di.sms), Cfg::kThreads, smem, stream>>>(prm);
    return launch_status();
}

// The bulk-copy path needs 16-byte aligned class rows (bases 16-byte aligned, pixels_per_image % 4 == 0).
inline bool tma_eligible(const FuseParams& prm) {
    if (prm.hw % 4 != 0) return false;
    for (int s = 0; s < prm.S; ++s)
        if (!aligned_to(prm.main[s], 16) || !aligned_to(prm.aux[s], 16) || (prm.kld[s] && !aligned_to(prm.kld[s], 16))) return false;
    return aligned_to(prm.label, 4) && (!prm.conf || aligned_to(prm.conf, 16)) && (!prm.unc || aligned_to(prm.unc, 16));
}

// ---- K1-lowres ------------------------------------------------------------------------------------------------------
// Fills prm.lr's stage layout for tiles of `tile_pix` consecutive output pixels; returns the dynamic shared memory the
// kernel needs with `stages` ring slots, or 0 if the geometry is unsupported (rows not 16-byte multiples).
inline size_t lowres_plan(FuseParams& prm, int tile_pix, int chunk, int stages, int KT, int nthreads, int P, int fixed_main = 0,
                          int fixed_aux = 0) {
    LowresGeom& lr = prm.lr;
    const int rows_spanned = (int)std::min<int64_t>(lr.H, (tile_pix - 1) / lr.W + 2);
    int main_stride = 0, aux_stride = 0;
    for (int s = 0; s < prm.S; ++s) {
        if (lr.wm[s] % 4 || lr.wa[s] % 4 || lr.hm[s] < 1 || lr.ha[s] < 1) return 0;
        auto rows = [&](int hin) {
            const float scale = lr.H > 1 ? (float)(hin - 1) / (float)(lr.H - 1) : 0.f;
            return std::min(hin, (int)((rows_spanned - 1) * scale) + 3);
        };
        main_stride = std::max(main_stride, rows(lr.hm[s]) * lr.wm[s]);
        aux_stride = std::max(aux_stride, rows(lr.ha[s]) * lr.wa[s]);
    }
    if (fixed_main > 0 && fixed_aux > 0) {          // compile-time strides requested: they must cover the geometry
        if (main_stride + 1 > fixed_main || aux_stride + 1 > fixed_aux) return 0;      // (+1: the taps' one-float overread)
        main_stride = fixed_main;
        aux_stride = fixed_aux;
    }
    else {                                           // the taps read one float past a row (PackedTaps): keep it inside the block
        main_stride += 4;
        aux_stride += 4;
    }
    lr.main_cls_stride = main_stride;
    lr.aux_cls_stride = aux_stride;
    lr.aux_base = chunk * main_stride;
    lr.stage_floats = chunk * (main_stride + aux_stride);
    lr.same_geometry = 1;
    for (int s = 1; s < prm.S; ++s)
        if (lr.hm[s] != lr.hm[0] || lr.wm[s] != lr.wm[0] || lr.ha[s] != lr.ha[0] || lr.wa[s] != lr.wa[0]) lr.same_geometry = 0;
    return sizeof(float) * (size_t)lr.stage_floats * stages + 2 * stages * sizeof(uint64_t) +
           fuse_tally_smem_bytes(prm.K, KT, nthreads, P) + 128;
}

}  // namespace mspl
