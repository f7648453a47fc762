// Host entry points for K1 (mspl_fuse_sources) and the hard-label vote (mspl_vote_labels).
#include <cstdio>
#include <cstring>

#include "fuse_launch.cuh"

namespace mspl {

// TMA-staged kernel configuration <consumer warps, pixels per thread, classes per chunk, ring stages>, picked from the
// tools/k1_sweep runs on B200 (profiles/): 15 consumer + 1 producer warps = 16 warps, so the register file splits evenly
// (128 regs/thread); 960-pixel tiles, 4 x 38.4 KB stages.  Since round 2 every policy runs this one shape: with the classes
// visited grouped by target the per-target maxima cost nothing extra per class (pixel_math.cuh), so 'half' / 'prob' differ
// from 'all' only in the per-source epilogue.  More than 5 target classes: 3 stages (their histogram and group slots need
// the shared memory of the fourth).
template <int KT> constexpr int kTmaStages = KT <= 5 ? 4 : 3;
constexpr int kDirectThreads = 256;
constexpr int kDirectMinBlocks = 2;     // direct kernel without GK: resident CTAs per SM the register allocator must leave room for
// K1-lowres: 15 consumer warps (instruction-bound kernel; 16 warps split the register file evenly), 4 ring stages
constexpr int kLowresNcw = 15, kLowresStages = 4;

template <int KT>
static int dispatch_fuse(FuseParams& prm, bool gk, cudaStream_t stream) {
    constexpr int CH = kFuseChunk, NST = kTmaStages<KT>;
    using Cfg = TmaCfg<15, 2, CH, NST>;
    if (!build_class_order(prm, CH)) return MSPL_ERR_UNSUPPORTED;
    if (tma_eligible(prm)) {
        const size_t smem = Cfg::smem_bytes(prm.K, KT);
        // nothing but hard labels requested under a vote policy (the reference's own generation loop): no softmax at all
        const bool labels_only = prm.policy == MSPL_POLICY_VOTE && !prm.conf && !prm.unc && !prm.conf_hist && !prm.marginal;
        bool any_kld = false;
        for (int s = 0; s < prm.S; ++s) any_kld = any_kld || prm.kld[s] != nullptr;
        if (labels_only && !any_kld) return launch_fuse_ring<Cfg>(fuse_labels_tma_kernel<15, 2, CH, NST, KT>, prm, smem, stream);
        if (gk) return launch_fuse_ring<Cfg>(fuse_sources_tma_kernel<15, 2, CH, NST, KT, true>, prm, smem, stream);
        return launch_fuse_ring<Cfg>(fuse_sources_tma_kernel<15, 2, CH, NST, KT, false>, prm, smem, stream);
    }
    // odd shapes / unaligned views: per-thread scalar streaming loads, same math
    if (gk) return launch_fuse_direct<kDirectThreads>(fuse_sources_direct_kernel<CH, KT, true, kDirectThreads, 1>, prm, KT, stream);
    return launch_fuse_direct<kDirectThreads>(fuse_sources_direct_kernel<CH, KT, false, kDirectThreads, kDirectMinBlocks>, prm, KT,
                                              stream);
}

// merge_outputs (uest_seg_multi_os.py:695-718) on (S, npix) hard labels.
__global__ void __launch_bounds__(256) vote_labels_kernel(const uint8_t* __restrict__ labels, int S, int64_t npix, int K,
                                                          int vote_t, int ignore, uint8_t* __restrict__ merged) {
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < npix; i += (int64_t)gridDim.x * blockDim.x) {
        uint32_t votes = 0;
        for (int s = 0; s < S; ++s) {
            const uint32_t l = labels[s * npix + i];
            if (l < (uint32_t)K) votes += 1u << (4 * l);   // values outside [0,K) match no class_id, as in the reference
        }
        merged[i] = (uint8_t)merge_votes<MSPL_MAX_CLASSES>(votes, vote_t, ignore);
    }
}

}  // namespace mspl

using namespace mspl;

extern "C" const char* mspl_fuse_variant(void) {
    static char name[256];
    snprintf(name, sizeof(name),
             "tma-bulk ring, CH=%d, classes visited grouped by target, packed f32x2 math: <15 consumer warps, P=2, 4 stages> for "
             "every policy; direct-ldg P=1 fallback for unaligned shapes",
             kFuseChunk);
    return name;
}

// Host-only: the class visiting order K1 derives from a label table (no device work; lets the host logic be tested on CPU).
// The class order K1 builds for one source with label table `lut`, into prm.order[0]; MSPL_OK or a negative status.
static int class_order_of_table(const uint8_t* lut, int num_classes, int num_target_classes, FuseParams& prm) {
    if (!lut || num_classes < 1 || num_classes > MSPL_MAX_SRC_CLASSES) return MSPL_ERR_BAD_ARG;
    if (num_target_classes < 2 || num_target_classes > MSPL_MAX_CLASSES) return MSPL_ERR_BAD_ARG;
    memset(&prm, 0, sizeof(prm));
    prm.S = 1;
    prm.C[0] = num_classes;
    for (int c = 0; c < num_classes; ++c) {
        if (lut[c] >= num_target_classes) return MSPL_ERR_BAD_ARG;
        prm.lut[0][c] = lut[c];
    }
    return build_class_order(prm, kFuseChunk) ? MSPL_OK : MSPL_ERR_UNSUPPORTED;
}

extern "C" int mspl_class_order(const uint8_t* lut, int num_classes, int num_target_classes, uint8_t* row, uint8_t* seg,
                                uint32_t* present) {
    if (!row || !seg || !present) return MSPL_ERR_BAD_ARG;
    FuseParams prm;
    const int rc = class_order_of_table(lut, num_classes, num_target_classes, prm);
    if (rc != MSPL_OK) return rc;
    memcpy(row, prm.order[0].row, (size_t)num_classes);
    memcpy(seg, prm.order[0].seg, (size_t)((num_classes + kFuseChunk - 1) / kFuseChunk));
    *present = prm.order[0].present;
    return kFuseChunk;
}

extern "C" int mspl_class_order_votes(const uint8_t* lut, int num_classes, int num_target_classes, uint32_t* vote, uint32_t* nchunk) {
    if (!vote || !nchunk) return MSPL_ERR_BAD_ARG;
    FuseParams prm;
    const int rc = class_order_of_table(lut, num_classes, num_target_classes, prm);
    if (rc != MSPL_OK) return rc;
    memcpy(vote, prm.order[0].vote, sizeof(prm.order[0].vote));
    *nchunk = prm.order[0].nchunk;
    return (int)prm.order[0].ngroup;
}

extern "C" int mspl_class_order_shape(const uint8_t* lut, int num_classes, int num_target_classes) {
    FuseParams prm;
    const int rc = class_order_of_table(lut, num_classes, num_target_classes, prm);
    return rc != MSPL_OK ? rc : (int)prm.order[0].shape;
}

// Checks and copies into prm what both K1 entry points take, returning MSPL_OK or the status the entry point returns.  With no
// images (prm.n_img == 0) the sources are not looked at.  main_hw / aux_hw: K1-lowres's head sizes, nullptr at full resolution;
// K1-lowres also needs 16-byte aligned logits, KLD maps, confidences and uncertainties and hw % 4 == 0.  The checks run in a
// fixed order: of several bad arguments, the first one checked decides the status.
static int fuse_args(FuseParams& prm, int S, const float* const* main_logits, const float* const* aux_logits, const int* num_classes,
                     const uint8_t* const* lut, const int* main_hw, const int* aux_hw, int64_t num_images, int64_t hw, int K,
                     int policy, int vote_t, int ignore_label, int ds_rate, uint8_t* label, float* conf, float* unc,
                     float* const* kld_per_source, unsigned long long* class_hist, unsigned long long* conf_hist,
                     unsigned long long* marginal_count) {
    const bool lowres = main_hw != nullptr;
    if (S < 1 || S > MSPL_MAX_SOURCES || K < 2 || K > MSPL_MAX_CLASSES) return MSPL_ERR_BAD_ARG;
    if (!main_logits || !aux_logits || !num_classes || !lut || !label || !class_hist) return MSPL_ERR_BAD_ARG;
    if (num_images < 0 || ds_rate < 1) return MSPL_ERR_BAD_ARG;
    if (ignore_label < 0 || ignore_label >= K) return MSPL_ERR_BAD_ARG;
    if (policy != MSPL_POLICY_VOTE && policy != MSPL_POLICY_PROB) return MSPL_ERR_BAD_ARG;
    if (conf_hist && !conf) return MSPL_ERR_BAD_ARG;
    memset(&prm, 0, sizeof(prm));
    if (num_images == 0) return MSPL_OK;
    if (lowres && hw % 4 != 0) return MSPL_ERR_UNSUPPORTED;
    const size_t align = lowres ? 16 : 4;      // the direct kernel reads logits one float at a time
    for (int s = 0; s < S; ++s) {
        const int C = num_classes[s];
        if (C < 1 || C > MSPL_MAX_SRC_CLASSES || !main_logits[s] || !aux_logits[s] || !lut[s]) return MSPL_ERR_BAD_ARG;
        if (lowres) {
            if (main_hw[2 * s] < 1 || main_hw[2 * s + 1] < 1 || aux_hw[2 * s] < 1 || aux_hw[2 * s + 1] < 1) return MSPL_ERR_BAD_ARG;
            prm.lr.hm[s] = main_hw[2 * s]; prm.lr.wm[s] = main_hw[2 * s + 1];
            prm.lr.ha[s] = aux_hw[2 * s]; prm.lr.wa[s] = aux_hw[2 * s + 1];
        }
        if (!aligned_to(main_logits[s], align) || !aligned_to(aux_logits[s], align)) return MSPL_ERR_ALIGN;
        prm.main[s] = main_logits[s];
        prm.aux[s] = aux_logits[s];
        prm.kld[s] = kld_per_source ? kld_per_source[s] : nullptr;
        if (lowres && prm.kld[s] && !aligned_to(prm.kld[s], 16)) return MSPL_ERR_ALIGN;
        prm.C[s] = C;
        for (int c = 0; c < C; ++c) {
            if (lut[s][c] >= K) return MSPL_ERR_BAD_ARG;
            prm.lut[s][c] = lut[s][c];
        }
    }
    if ((lowres && !aligned_to(label, 4)) || (conf && !aligned_to(conf, align)) || (unc && !aligned_to(unc, align)))
        return MSPL_ERR_ALIGN;
    if (!aligned_to(class_hist, 8) || (conf_hist && !aligned_to(conf_hist, 8)) || (marginal_count && !aligned_to(marginal_count, 8)))
        return MSPL_ERR_ALIGN;
    prm.S = S; prm.K = K; prm.policy = policy; prm.vote_t = vote_t < 1 ? 1 : vote_t;
    prm.ignore = ignore_label; prm.ds_rate = ds_rate;
    prm.n_img = num_images; prm.hw = hw;
    prm.label = label; prm.conf = conf; prm.unc = unc;
    prm.class_hist = class_hist; prm.conf_hist = conf_hist; prm.marginal = marginal_count;
    return MSPL_OK;
}

// Per-target-class probabilities are only needed when a pixel can win without every source's vote.
// (under a vote policy they only ever feed conf, so a call without conf does not need them either)
static bool needs_target_probs(const FuseParams& prm) {
    return prm.policy == MSPL_POLICY_PROB || (prm.vote_t < prm.S && prm.conf != nullptr);
}

extern "C" int mspl_fuse_sources(int num_sources, const float* const* main_logits, const float* const* aux_logits,
                                 const int* num_classes, const uint8_t* const* lut, int64_t num_images,
                                 int64_t pixels_per_image, int num_target_classes, int policy, int vote_t,
                                 int ignore_label, int ds_rate, uint8_t* label, float* conf, float* unc,
                                 float* const* kld_per_source, unsigned long long* class_hist,
                                 unsigned long long* conf_hist, unsigned long long* marginal_count, void* stream) {
    if (pixels_per_image < 1) return MSPL_ERR_BAD_ARG;
    FuseParams prm;
    const int rc = fuse_args(prm, num_sources, main_logits, aux_logits, num_classes, lut, nullptr, nullptr, num_images,
                             pixels_per_image, num_target_classes, policy, vote_t, ignore_label, ds_rate, label, conf, unc,
                             kld_per_source, class_hist, conf_hist, marginal_count);
    if (rc != MSPL_OK || prm.n_img == 0) return rc;
    const bool gk = needs_target_probs(prm);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    return prm.K <= 5 ? dispatch_fuse<5>(prm, gk, st) : dispatch_fuse<8>(prm, gk, st);
}

extern "C" int mspl_fuse_sources_lowres(int num_sources, const float* const* main_logits, const float* const* aux_logits,
                                        const int* num_classes, const uint8_t* const* lut, const int* main_hw, const int* aux_hw,
                                        int64_t num_images, int out_h, int out_w, int num_target_classes, int policy, int vote_t,
                                        int ignore_label, int ds_rate, uint8_t* label, float* conf, float* unc,
                                        float* const* kld_per_source, unsigned long long* class_hist,
                                        unsigned long long* conf_hist, unsigned long long* marginal_count, void* stream) {
    if (!main_hw || !aux_hw || out_h < 1 || out_w < 1) return MSPL_ERR_BAD_ARG;
    FuseParams prm;
    const int rc = fuse_args(prm, num_sources, main_logits, aux_logits, num_classes, lut, main_hw, aux_hw, num_images,
                             (int64_t)out_h * out_w, num_target_classes, policy, vote_t, ignore_label, ds_rate, label, conf, unc,
                             kld_per_source, class_hist, conf_hist, marginal_count);
    if (rc != MSPL_OK || prm.n_img == 0) return rc;
    prm.lr.H = out_h; prm.lr.W = out_w;

    constexpr int NCW = kLowresNcw, P = 2, CH = kFuseChunk, NST = kLowresStages;
    using Cfg = TmaCfg<NCW, P, CH, NST>;
    const bool gk = needs_target_probs(prm);
    const int K = prm.K;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (!build_class_order(prm, CH)) return MSPL_ERR_UNSUPPORTED;
    if (K <= 5) {   // common geometries (e.g. ESPDNetUE at 480x256: 3 rows x 240 / 3 rows x 120 floats per class) fit fixed class
                    // strides, which turn every interpolation tap into an immediate-offset shared-memory load
        constexpr int MS = 768, AS = 384;
        FuseParams fixed = prm;
        const size_t fsmem = lowres_plan(fixed, Cfg::kTilePix, CH, NST, 5, Cfg::kThreads, P, MS, AS);
        if (fsmem != 0 && fsmem <= 227 * 1024) {
            if (gk) return launch_fuse_ring<Cfg>(fuse_sources_lowres_kernel<NCW, P, CH, NST, 5, true, MS, AS>, fixed, fsmem, st);
            return launch_fuse_ring<Cfg>(fuse_sources_lowres_kernel<NCW, P, CH, NST, 5, false, MS, AS>, fixed, fsmem, st);
        }
    }
    const int KT = K <= 5 ? 5 : 8;
    const size_t smem = lowres_plan(prm, Cfg::kTilePix, CH, NST, KT, Cfg::kThreads, P);
    if (smem == 0 || smem > 227 * 1024) return MSPL_ERR_UNSUPPORTED;    // caller upsamples and uses mspl_fuse_sources instead
    if (K <= 5) {
        if (gk) return launch_fuse_ring<Cfg>(fuse_sources_lowres_kernel<NCW, P, CH, NST, 5, true>, prm, smem, st);
        return launch_fuse_ring<Cfg>(fuse_sources_lowres_kernel<NCW, P, CH, NST, 5, false>, prm, smem, st);
    }
    if (gk) return launch_fuse_ring<Cfg>(fuse_sources_lowres_kernel<NCW, P, CH, NST, 8, true>, prm, smem, st);
    return launch_fuse_ring<Cfg>(fuse_sources_lowres_kernel<NCW, P, CH, NST, 8, false>, prm, smem, st);
}

extern "C" int mspl_vote_labels(const uint8_t* labels, int num_sources, int64_t num_pixels, int num_target_classes,
                                int vote_t, int ignore_label, uint8_t* merged, void* stream) {
    if (!labels || !merged || num_sources < 1 || num_sources > 15 || num_pixels < 0) return MSPL_ERR_BAD_ARG;
    if (num_target_classes < 1 || num_target_classes > MSPL_MAX_CLASSES) return MSPL_ERR_BAD_ARG;
    if (num_pixels == 0) return MSPL_OK;
    int64_t blocks = (num_pixels + 255) / 256;
    if (blocks > kNumSMs * 16) blocks = kNumSMs * 16;
    vote_labels_kernel<<<(unsigned)blocks, 256, 0, static_cast<cudaStream_t>(stream)>>>(
        labels, num_sources, num_pixels, num_target_classes, vote_t, ignore_label, merged);
    return launch_status();
}
