// K1 -- fused multi-source pseudo-label generation.
//
// One pass over HBM: every (main, aux) logit of every source is read exactly once; per pixel the kernel produces the
// voted / fused label (u8), its confidence, the mean main-vs-aux KLD, and accumulates the class histogram plus the linear
// per-class confidence histogram in shared memory.  Replaces uest_seg_multi_os.py:897-921 (+ :669-718)
// -- see include/mspl_b200.h.
//
// Two load mechanisms share all the per-pixel math (pixel_math.cuh):
//   fuse_sources_direct_kernel : every thread streams its own pixel with ld.global.nc (any shape / alignment)
//   fuse_sources_tma_kernel    : a producer warp stages [classes-chunk x tile-of-pixels] boxes into a shared-memory
//                                ring with bulk async copies (TMA engine, cp.async.bulk + mbarrier complete_tx),
//                                consumer warps compute from shared memory; bytes in flight no longer cost registers
// Both visit a source's classes grouped by target class (ClassOrder), see pixel_math.cuh.
#pragma once
#include <type_traits>
#include <utility>

#include "pixel_math.cuh"
#include "bilinear.cuh"

namespace mspl {

// Geometry of the fused-upsample variant (K1-lowres): the sources hand over their logits BEFORE the network's final
// F.interpolate(..., mode='bilinear', align_corners=True) (model/segmentation/espdnet_ue.py:301-302); the kernel
// interpolates on the fly.  All zero for the plain kernels.
struct LowresGeom {
    int H, W;                            // output (full) resolution; hw == H * W
    int hm[MSPL_MAX_SOURCES], wm[MSPL_MAX_SOURCES];   // main head resolution per source
    int ha[MSPL_MAX_SOURCES], wa[MSPL_MAX_SOURCES];   // aux head resolution per source
    int main_cls_stride, aux_cls_stride, aux_base;    // float offsets inside one ring stage
    int stage_floats;
    int same_geometry;                                // every source has the head sizes of source 0
};

struct FuseParams {
    const float* main[MSPL_MAX_SOURCES];
    const float* aux[MSPL_MAX_SOURCES];
    float* kld[MSPL_MAX_SOURCES];
    int C[MSPL_MAX_SOURCES];
    uint8_t lut[MSPL_MAX_SOURCES][MSPL_MAX_SRC_CLASSES];
    ClassOrder order[MSPL_MAX_SOURCES];
    int S, K, policy, vote_t, ignore, ds_rate;
    int64_t n_img, hw;
    uint8_t* label;
    float* conf;
    float* unc;
    unsigned long long* class_hist;
    unsigned long long* conf_hist;
    unsigned long long* marginal;
    LowresGeom lr;
};

// Shared-memory bookkeeping common to all kernels:
//   [K*2048 u32 conf histogram][16 u32: class counts + spare][S*256 B label tables][S*256 B class visiting order][16 B slack]
//   [KT * nthreads * P floats: committed group maxima, one column per thread]
inline size_t fuse_tally_smem_bytes(int K, int KT, int nthreads, int P) {
    size_t b = sizeof(uint32_t) * ((size_t)K * MSPL_RADIX_BINS + 16) + 2 * MSPL_MAX_SOURCES * MSPL_MAX_SRC_CLASSES + 16;
    b = (b + 15) & ~(size_t)15;
    return b + sizeof(float) * (size_t)KT * nthreads * P;
}

// merge_outputs (uest_seg_multi_os.py:695-718) on one pixel's packed vote counters (4 bits per target class; classes from
// the call's K up to KT carry no votes): the class with the most votes, the lowest one on ties (:713), and `ignore` when it
// has fewer than vote_t votes (:716).
template <int KT>
MSPL_DEVINL int merge_votes(uint32_t votes, int vote_t, int ignore) {
    int bk = 0;
    uint32_t bc = votes & 15u;
#pragma unroll
    for (int k = 1; k < KT; ++k) {
        const uint32_t c = (votes >> (4 * k)) & 15u;
        if (c > bc) { bc = c; bk = k; }
    }
    return ((int)bc < vote_t) ? ignore : bk;
}

// ---- per-pixel accumulation across sources --------------------------------------------------------------------------
// GK: per-target-class probabilities needed (policy 'prob', or a vote threshold below S); otherwise every source voted
// for the winning label and G_s[label] is simply that source's max probability.
template <int P, int K, bool GK>
struct PixelFusion {
    Px<P> usum, csum, Fk[GK ? K : 1];
    Px<P> mgap;             // min over the sources of (z_best - z_runner-up) * pmax: the near-tie report
    uint32_t votes[P];      // 4 bits per target class
    uint32_t last_vote[P];  // what the most recent source added (1 << 4*label): unanimity shortcut in finish()
    bool marg[P];           // set by finish()

    MSPL_DEVINL void reset() {
        usum = csum = Px<P>::splat(0.f);
        mgap = Px<P>::splat(INFINITY);
#pragma unroll
        for (int k = 0; k < (GK ? K : 1); ++k) Fk[k] = Px<P>::splat(0.f);
#pragma unroll
        for (int p = 0; p < P; ++p) votes[p] = 0;
    }

    // Fold one finished source in; d receives its KLD map values.  group: this thread's column of committed group maxima
    // (g = max z over the source classes mapped to one target; committed in ascending target order, one entry per target the
    // source's table maps to at all).
    // slow: the kernel's out-of-line recomputations, slow.pmax(p, Mz) for a degenerate pixel and slow.label(p) for an exact
    // tie between two targets (only those touch global memory again).
    template <typename Slow>
    MSPL_DEVINL void add_source(const SourceStats<P>& st, const Px<P>* group, int gstride, const ClassOrder& order, float (&d)[P], Slow slow) {
        // the source's proposal: the target whose group holds the largest z; the runner-up target gives the near-tie
        // report and detects exact ties between targets (those are resolved out of line, so the scan order is free)
        Px<P> gp[K];
        float best[P], second[P];
        uint32_t vote[P];
        if (GK) {
            // per-target probabilities are needed below: one value per TARGET, -inf for targets the table never maps to
            const uint32_t present = order.present;
            float g[K][P];
            const Px<P>* next = group;
#pragma unroll
            for (int k = 0; k < K; ++k) {
                if ((present >> k) & 1u) {
                    gp[k] = *next;
                    next += gstride;
                } else {
                    gp[k] = Px<P>::splat(-INFINITY);
                }
                gp[k].get(g[k]);
            }
#pragma unroll
            for (int p = 0; p < P; ++p) {
                best[p] = g[0][p];
                second[p] = -INFINITY;
                vote[p] = 1u;
#pragma unroll
                for (int k = 1; k < K; ++k) {
                    second[p] = fmaxf(second[p], fminf(best[p], g[k][p]));
                    vote[p] = (g[k][p] > best[p]) ? (1u << (4 * k)) : vote[p];
                    best[p] = fmaxf(best[p], g[k][p]);
                }
            }
        } else {
            // only the winner matters: scan the committed groups themselves (ngroup <= K of them, a warp-uniform count) and
            // take the winner's vote increment from the order's table.  All K entries of the column are loaded up front
            // (those past ngroup are stale and never looked at), so the loads overlap instead of trailing the branches.
            const int ngroup = (int)order.ngroup;
#pragma unroll
            for (int i = 0; i < K; ++i) gp[i] = Px<P>::load_shared_now(group + i * gstride);
            gp[0].get(best);
#pragma unroll
            for (int p = 0; p < P; ++p) vote[p] = order.vote[0];
#pragma unroll
            for (int i = 1; i < K; ++i) {
                if (i < ngroup) {
                    float gi[P];
                    gp[i].get(gi);
                    const uint32_t vi = order.vote[i];
#pragma unroll
                    for (int p = 0; p < P; ++p) {
                        const float lo = fminf(best[p], gi[p]);
                        second[p] = (i == 1) ? lo : fmaxf(second[p], lo);
                        vote[p] = (gi[p] > best[p]) ? vi : vote[p];
                        best[p] = fmaxf(best[p], gi[p]);
                    }
                } else if (i == 1) {
#pragma unroll
                    for (int p = 0; p < P; ++p) second[p] = -INFINITY;       // a single group: no runner-up
                }
            }
        }
        const Px<P> Mz = Px<P>::make(best);
        SourceResult<P> r = finish_source<P>(st, Mz);
        float gap[P];
        r.gap.get(gap);
        bool slow_any = false;
#pragma unroll
        for (int p = 0; p < P; ++p) slow_any |= degenerate_source(gap[p], best[p]) | (second[p] == best[p]);
        if (slow_any) {       // ONE rare, divergent region for both out-of-line recomputations of all the thread's pixels
            float rz[P], inv_sz[P], pm[P];
            r.rz.get(rz); r.inv_sz.get(inv_sz); r.pmax.get(pm);
#pragma unroll
            for (int p = 0; p < P; ++p) {
                if (degenerate_source(gap[p], best[p])) {
                    rz[p] = best[p];
                    inv_sz[p] = pm[p] = slow.pmax(p, best[p]);
                }
                // first maximal class in ORIGINAL order decides (np.argmax, :904)
                if (second[p] == best[p]) vote[p] = 1u << (4 * slow.label(p));
            }
            r.rz = Px<P>::make(rz); r.inv_sz = Px<P>::make(inv_sz); r.pmax = Px<P>::make(pm);
        }
        r.kld.get(d);
        usum = usum + r.kld;
        // near-tie report: P_best - P_runner-up = pmax * (1 - e^{-(best - second)}) < 1e-6.  The gap that satisfies it is at
        // most 1e-6 / pmax <= 2.6e-4 (pmax >= 1/256), where 1 - e^{-x} = x to a relative 1.3e-4: the exponential is not needed.
        // (finish() compares the minimum over the sources; a NaN product -- both -inf -- never lowers it.)
        mgap = pmin<P>(mgap, (Mz - Px<P>::make(second)) * r.pmax);
#pragma unroll
        for (int p = 0; p < P; ++p) {
            votes[p] += vote[p];
            last_vote[p] = vote[p];
        }
        if (GK) {
            const Px<P> l2e = Px<P>::splat(kLog2e), one = Px<P>::splat(1.0f);
#pragma unroll
            for (int k = 1; k < K; ++k)      // G[0] = 0 as transfer_output_to_greenhouse (uest_seg_multi_os.py:1340)
                Fk[GK ? k : 0] = Fk[GK ? k : 0] + pmin<P>(pex2<P>((gp[k] - r.rz) * l2e) * r.inv_sz, one);
        } else {
            csum = csum + r.pmax;
        }
    }

    // inv_s = 1/S: the averages over sources are formed as sum * (1/S) (one rounding away from the sum / S the
    // definition states; far inside the 1e-5 tolerance) to keep IEEE division sequences out of the hot loop
    MSPL_DEVINL void finish(const FuseParams& prm, float inv_s, int (&label)[P], float (&conf)[P], float (&unc)[P]) {
        const int ignore = prm.ignore;
        float us[P], cs[P], fk[GK ? K : 1][P], mg[P];
        usum.get(us); csum.get(cs); mgap.get(mg);
#pragma unroll
        for (int k = 0; k < (GK ? K : 1); ++k) Fk[k].get(fk[k]);
#pragma unroll
        for (int p = 0; p < P; ++p) {
            unc[p] = us[p] * inv_s;
            marg[p] = mg[p] < kNearTieMargin;
            if (prm.policy == MSPL_POLICY_PROB) {
                float best = -1.f, second = -1.f;
                int bk = 0;
#pragma unroll
                for (int k = 0; k < K; ++k) {
                    const float f = GK ? fk[GK ? k : 0][p] * inv_s : 0.f;
                    second = fmaxf(second, fminf(best, f));
                    bk = (f > best) ? k : bk;
                    best = fmaxf(best, f);
                }
                label[p] = bk;
                conf[p] = best;
                marg[p] |= (best - second) < kNearTieMargin;
            } else {
                if (!GK && prm.vote_t == prm.S) {
                    // unanimity required ('all'): the label survives only if every source proposed it, so looking at the
                    // last proposal's count is enough -- no scan over the classes
                    const int bk = (31 - __clz((int)last_vote[p])) >> 2;
                    label[p] = ((int)((votes[p] >> (4 * bk)) & 15u) < prm.vote_t) ? ignore : bk;
                } else {
                    label[p] = merge_votes<K>(votes[p], prm.vote_t, ignore);
                }
                // every source voted for `label`, so G_s[label] is that source's max probability -- except for target class 0,
                // which transfer_output_to_greenhouse never fills (G[0] = 0, uest_seg_multi_os.py:1340)
                float f = (label[p] == 0) ? 0.f : cs[p];
                if (GK) {
                    // F[label] by masking (a select chain over k gets turned into an indexed load of Fk from LOCAL memory)
                    uint32_t bits = 0;
#pragma unroll
                    for (int k = 0; k < K; ++k) bits |= __float_as_uint(fk[GK ? k : 0][p]) & (0u - (uint32_t)(label[p] == k));
                    f = __uint_as_float(bits);
                }
                conf[p] = (label[p] == ignore) ? 0.f : f * inv_s;
            }
        }
    }
};

// ---- per-thread tallies: class counts (packed 8 bits per class, spilled before overflow), near-ties, histogram ----------
template <int K>
struct Tally {
    unsigned long long packed = 0;
    uint32_t full[K] = {};
    uint32_t n_marginal = 0, n_ignore_zero = 0;
    int pending = 0;

    MSPL_DEVINL void spill() {
#pragma unroll
        for (int k = 0; k < K; ++k) full[k] += (uint32_t)(packed >> (8 * k)) & 0xffu;
        packed = 0;
        pending = 0;
    }

    template <int P>
    MSPL_DEVINL void add(const FuseParams& prm, uint32_t* s_hist, const int (&label)[P], const float (&conf)[P],
                         const bool (&marg)[P], int64_t off, bool active) {
        const bool want_hist = prm.conf_hist != nullptr;
#pragma unroll
        for (int p = 0; p < P; ++p) {
            packed += (unsigned long long)active << (8 * label[p]);
            n_marginal += (marg[p] && active);
            if (want_hist) {
                const bool keep = active && (prm.ds_rate <= 1 || ((off + p) % prm.ds_rate) == 0);
                // vote policies give ignore-labelled pixels conf == 0: one known bin, counted without atomics
                if (prm.policy != MSPL_POLICY_PROB && label[p] == prm.ignore) n_ignore_zero += keep;
                else if (keep) atomicAdd(&s_hist[label[p] * MSPL_RADIX_BINS + conf_bin(conf[p])], 1u);
            }
        }
        if ((pending += P) > 255 - P) spill();
    }

    // whole CTA must call this (it syncs); nthreads = blockDim.x
    MSPL_DEVINL void flush(const FuseParams& prm, uint32_t* s_hist, uint32_t* s_cls, int nthreads) {
        spill();
        const bool leader = (threadIdx.x & 31) == 0;
#pragma unroll
        for (int k = 0; k < K; ++k) {
            const uint32_t w = __reduce_add_sync(0xffffffffu, full[k]);
            if (leader && w) atomicAdd(&s_cls[k], w);
        }
        const uint32_t wz = __reduce_add_sync(0xffffffffu, n_ignore_zero);
        if (leader && wz) atomicAdd(&s_hist[prm.ignore * MSPL_RADIX_BINS + conf_bin(0.f)], wz);
        const uint32_t wm = __reduce_add_sync(0xffffffffu, n_marginal);
        if (leader && wm && prm.marginal) atomicAdd(prm.marginal, (unsigned long long)wm);
        __syncthreads();
        if ((int)threadIdx.x < prm.K && s_cls[threadIdx.x]) atomicAdd(prm.class_hist + threadIdx.x, (unsigned long long)s_cls[threadIdx.x]);
        if (prm.conf_hist)
            for (int i = threadIdx.x; i < prm.K * MSPL_RADIX_BINS; i += nthreads)
                if (s_hist[i]) atomicAdd(prm.conf_hist + i, (unsigned long long)s_hist[i]);
    }
};

// End of a tile for the thread's P pixels off, off + 1, ... of image n (hw pixels per image): the fused label, conf and unc to
// global memory (active: the pixels exist), then into the tallies.  inv_s = 1/S.
template <int P, int KT, bool GK>
MSPL_DEVINL void finish_tile(const FuseParams& prm, PixelFusion<P, KT, GK>& fus, float inv_s, Tally<KT>& tally, uint32_t* s_hist,
                             int64_t n, int64_t hw, int64_t off, bool active) {
    int label[P];
    float conf[P], unc[P];
    fus.finish(prm, inv_s, label, conf, unc);
    if (active) {
        const int64_t o = n * hw + off;
        store_labels<P>(prm.label + o, label);
        if (prm.conf) PixVec<P>::store(prm.conf + o, conf);
        if (prm.unc) PixVec<P>::store(prm.unc + o, unc);
    }
    tally.template add<P>(prm, s_hist, label, conf, fus.marg, off, active);
}

// Carves the bookkeeping region (layout: fuse_tally_smem_bytes) and initialises it; the caller syncs.
struct TallySmem {
    uint32_t* hist;
    uint32_t* cls;
    uint8_t* lut;       // [S][256] label tables (slow paths, labels-only kernel)
    uint8_t* row;       // [S][256] class visiting order
    float* group;       // [KT][nthreads][P]
};
// group_floats: size of the committed-maxima region ([KT][nthreads][P] floats), set to -inf so that no entry is ever read
// uninitialised (the epilogue loads all KT entries of a thread's column and ignores those its source did not commit).
MSPL_DEVINL TallySmem tally_smem_init(const FuseParams& prm, unsigned char* smem, int nthreads, int group_floats = 0) {
    TallySmem t;
    const int nbins = prm.K * MSPL_RADIX_BINS;
    t.hist = reinterpret_cast<uint32_t*>(smem);
    t.cls = t.hist + nbins;
    t.lut = reinterpret_cast<uint8_t*>(t.cls + 16);
    t.row = t.lut + MSPL_MAX_SOURCES * MSPL_MAX_SRC_CLASSES;
    size_t off = sizeof(uint32_t) * ((size_t)nbins + 16) + 2 * MSPL_MAX_SOURCES * MSPL_MAX_SRC_CLASSES + 16;
    off = (off + 15) & ~(size_t)15;
    t.group = reinterpret_cast<float*>(smem + off);
    for (int i = threadIdx.x; i < nbins; i += nthreads) t.hist[i] = 0;
    for (int i = threadIdx.x; i < group_floats; i += nthreads) t.group[i] = -INFINITY;
    if (threadIdx.x < 16) t.cls[threadIdx.x] = 0;
    for (int i = threadIdx.x; i < prm.S * MSPL_MAX_SRC_CLASSES; i += nthreads) {
        t.lut[i] = prm.lut[i / MSPL_MAX_SRC_CLASSES][i % MSPL_MAX_SRC_CLASSES];
        t.row[i] = prm.order[i / MSPL_MAX_SRC_CLASSES].row[i % MSPL_MAX_SRC_CLASSES];
    }
    return t;
}

// Slow paths of the full-resolution kernels: re-read the pixel's logits from global memory.  Only coordinates are kept; the
// pointers are formed inside the (rare) branch so that the common path pays nothing for them.
template <int P>
struct GlobalSlowPath {
    const FuseParams& prm;
    int s;
    int64_t n, off;       // image, this thread's first pixel inside it
    const uint8_t* lut;
    MSPL_DEVINL float pmax(int p, float Mz) const {
        const int64_t o = ((int64_t)n * prm.C[s]) * prm.hw + off + p;
        return recompute_pmax(prm.main[s] + o, prm.aux[s] + o, prm.C[s], prm.hw, Mz);
    }
    MSPL_DEVINL int label(int p) const {
        const int64_t o = ((int64_t)n * prm.C[s]) * prm.hw + off + p;
        return recompute_label(prm.main[s] + o, prm.aux[s] + o, prm.C[s], prm.hw, lut);
    }
};

// ======================================================================================================================
// Direct-load kernel (fallback for unaligned / odd shapes).  One pixel per thread, CH: classes per chunk, KT: compile-time
// bound on the target classes (prm.K <= KT; classes in [prm.K, KT) never receive votes or probability).
// ======================================================================================================================
template <int CH, int KT, bool GK, int THREADS, int MINB>
__global__ void __launch_bounds__(THREADS, MINB) fuse_sources_direct_kernel(const __grid_constant__ FuseParams prm) {
    constexpr int P = 1;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const TallySmem ts = tally_smem_init(prm, smem_raw, THREADS, KT * THREADS);
    __syncthreads();

    const int S = prm.S;
    const float fS = 1.0f / (float)S;
    const int64_t hw = prm.hw;
    const int64_t n_groups = prm.n_img * hw;
    const int64_t n_tiles = (n_groups + THREADS - 1) / THREADS;
    Tally<KT> tally;
    Px<P>* group = reinterpret_cast<Px<P>*>(ts.group) + threadIdx.x;

    for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        int64_t g = tile * THREADS + threadIdx.x;
        const bool active = g < n_groups;
        g = active ? g : n_groups - 1;
        const int64_t n = g / hw;
        const int64_t off = g - n * hw;

        PixelFusion<P, KT, GK> fus;
        fus.reset();
        for (int s = 0; s < S; ++s) {
            const int C = prm.C[s];
            const float* pm = prm.main[s] + (n * C) * hw + off;
            const float* pa = prm.aux[s] + (n * C) * hw + off;
            const uint8_t* row = ts.row + s * MSPL_MAX_SRC_CLASSES;
            SourceStats<P> st;
            st.reset(group);
            for (int c0 = 0; c0 < C; c0 += CH) {
                Px<P> m[CH], a[CH];
#pragma unroll
                for (int j = 0; j < CH; ++j) {
                    float mv[1] = {kPadLogit}, av[1] = {kPadLogit};
                    if (c0 + j < C) {
                        PixVec<1>::load(pm + (int64_t)row[c0 + j] * hw, mv);
                        PixVec<1>::load(pa + (int64_t)row[c0 + j] * hw, av);
                    }
                    m[j] = Px<P>::make(mv);
                    a[j] = Px<P>::make(av);
                }
                fold_chunk<P, CH>(st, m, a, c0 == 0, prm.order[s].seg[c0 / CH], THREADS);
            }
            float d[P];
            fus.add_source(st, group, THREADS, prm.order[s], d, GlobalSlowPath<P>{prm, s, n, off, ts.lut + s * MSPL_MAX_SRC_CLASSES});
            if (prm.kld[s] != nullptr && active) PixVec<P>::store(prm.kld[s] + n * hw + off, d);
        }
        finish_tile(prm, fus, fS, tally, ts.hist, n, hw, off, active);
    }
    tally.flush(prm, ts.hist, ts.cls, THREADS);
}

// ======================================================================================================================
// TMA (bulk async copy) staged kernel.
//   CTA = NCW consumer warps + 1 producer warp.  A tile is up to TP = NCW*32*P consecutive pixels of one image (the
//   last tile of an image may be shorter; hw % 4 == 0 keeps every row copy a multiple of 16 bytes).
//   A stage holds one chunk of up to CH classes of both heads for the tile: [2][CH][TP] floats; the producer fills stages
//   in the order (tile, source, chunk) with one cp.async.bulk per class row, completion signalled on the stage's "full"
//   mbarrier (complete_tx::bytes); a consumer warp copies its pixels' values to registers, releases the stage ("empty"
//   mbarrier, one arrival per consumer warp) and only then does the math, so the ring turns over at load speed.
// ======================================================================================================================
namespace tma {

MSPL_DEVINL uint32_t smem_addr(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

MSPL_DEVINL void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_addr(bar)), "r"(count) : "memory");
}
MSPL_DEVINL void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_addr(bar)) : "memory");
}
MSPL_DEVINL void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_addr(bar)), "r"(bytes) : "memory");
}
// Wait for a phase of `bar`.  try_wait suspends the warp in hardware up to a time limit before it has to be re-issued; the
// hint asks for a long suspension (the producer is HBM-bound: a stage takes ~1 us to fill), so that waiting warps do not burn
// issue slots -- and board power, which is what caps this kernel's sustained rate -- on a spin loop (6 % of all executed
// instructions without the hint, ncu source page of round 2).
constexpr uint32_t kMbarSuspendNs = 2000;
MSPL_DEVINL void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1, %2;\n"
        "@p bra DONE_%=;\n"
        "bra WAIT_%=;\n"
        "DONE_%=:\n"
        "}\n" ::"r"(smem_addr(bar)), "r"(parity), "r"(kMbarSuspendNs)
        : "memory");
}
// 1-D bulk copy global -> shared, completion counted in bytes on `bar`; streaming data: L2 evict-first hint
MSPL_DEVINL void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar, uint64_t policy) {
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;" ::"r"(smem_addr(dst)),
        "l"(src), "r"(bytes), "r"(smem_addr(bar)), "l"(policy)
        : "memory");
}
MSPL_DEVINL uint64_t evict_first_policy() {
    uint64_t p;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
    return p;
}

template <int P> MSPL_DEVINL void lds(const float* p, float (&v)[P]);
template <> MSPL_DEVINL void lds<1>(const float* p, float (&v)[1]) { v[0] = *p; }
template <> MSPL_DEVINL void lds<2>(const float* p, float (&v)[2]) {
    const float2 t = *reinterpret_cast<const float2*>(p);
    v[0] = t.x; v[1] = t.y;
}
template <> MSPL_DEVINL void lds<4>(const float* p, float (&v)[4]) {
    const float4 t = *reinterpret_cast<const float4*>(p);
    v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
}
// P pixels of one class row straight into the packed form
template <int P> MSPL_DEVINL Px<P> lds_px(const float* p) {
    float v[P];
    lds<P>(p, v);
    return Px<P>::make(v);
}

}  // namespace tma

template <int NCW, int P, int CH, int NSTAGE>
struct TmaCfg {
    static constexpr int kThreads = (NCW + 1) * 32;
    static constexpr int kTilePix = NCW * 32 * P;
    static constexpr int kStageFloats = 2 * CH * kTilePix;
    static constexpr size_t kRingBytes = sizeof(float) * (size_t)kStageFloats * NSTAGE;
    static size_t smem_bytes(int K, int KT) {
        return kRingBytes + 2 * NSTAGE * sizeof(uint64_t) + fuse_tally_smem_bytes(K, KT, kThreads, P) + 128;
    }
};

// The shared-memory ring of the staged kernels: NSTAGE slots of stage_floats floats, then one "full" and one "empty" mbarrier
// per slot,  [slots][full x NSTAGE][empty x NSTAGE].  The producer warp fills the slots in turn and the NCW consumer warps
// drain them in the same order; each thread's copy of this struct holds its own position (stage, phase) in that sequence.
template <int NCW, int NSTAGE>
struct StageRing {
    float* base;
    uint64_t* full;
    uint64_t* empty;
    int stage_floats;
    int stage = 0;
    uint32_t phase = 0;

    MSPL_DEVINL StageRing(unsigned char* smem, int stage_floats_)
        : base(reinterpret_cast<float*>(smem)), full(reinterpret_cast<uint64_t*>(smem + sizeof(float) * (size_t)stage_floats_ * NSTAGE)),
          empty(full + NSTAGE), stage_floats(stage_floats_) {}
    // first byte after the barriers
    MSPL_DEVINL unsigned char* end() const { return reinterpret_cast<unsigned char*>(empty + NSTAGE); }
    // "full" completes on the producer's arrival plus the bytes of its copies, "empty" on one arrival per consumer warp.  The
    // caller syncs the CTA before the ring is used.
    MSPL_DEVINL void init() const {
        if (threadIdx.x == 0) {
            for (int i = 0; i < NSTAGE; ++i) {
                tma::mbar_init(&full[i], 1);
                tma::mbar_init(&empty[i], NCW);
            }
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        }
    }
    MSPL_DEVINL float* slot() const { return base + (size_t)stage * stage_floats; }
    MSPL_DEVINL void advance() {
        if (++stage == NSTAGE) { stage = 0; phase ^= 1; }
    }
    // consumer: wait until the current slot is filled
    MSPL_DEVINL const float* wait_full() const {
        tma::mbar_wait(&full[stage], phase);
        return slot();
    }
    // consumer warp: its values are in registers, hand the slot back and move on
    MSPL_DEVINL void release(int lane) {
        __syncwarp();
        if (lane == 0) tma::mbar_arrive(&empty[stage]);
        advance();
    }
    // producer: wait until every consumer warp has released the current slot
    MSPL_DEVINL float* wait_empty() const {
        tma::mbar_wait(&empty[stage], phase ^ 1);
        return slot();
    }
    // producer warp: announce `bytes` of bulk copies into the current slot (a release: it publishes what the warp wrote into the
    // slot before, the padding); the copies complete on the returned barrier.  advance() once they are issued.
    MSPL_DEVINL uint64_t* expect(int lane, uint32_t bytes) const {
        __syncwarp();
        if (lane == 0) tma::mbar_arrive_expect_tx(&full[stage], bytes);
        return &full[stage];
    }
};

// Producer warp, tail chunk of cn < CH classes: the class rows the source does not have are filled with kPadLogit HERE, so that
// the consumers' loads and math carry no predicates and exist only once in the instruction stream.  n4: float4 per row of a
// head; stride: floats from one class row (block) of a head to the next; the aux head's rows start at aux_base.
template <int CH>
MSPL_DEVINL void pad_tail_rows(float* dst, int cn, int lane, int main_n4, int main_stride, int aux_base, int aux_n4, int aux_stride) {
    const float4 pad = make_float4(kPadLogit, kPadLogit, kPadLogit, kPadLogit);
    for (int j = cn; j < CH; ++j) {
        for (int i = lane; i < main_n4; i += 32) reinterpret_cast<float4*>(dst + j * main_stride)[i] = pad;
        for (int i = lane; i < aux_n4; i += 32) reinterpret_cast<float4*>(dst + aux_base + j * aux_stride)[i] = pad;
    }
    __threadfence_block();
}

// This CTA's tiles blockIdx.x, blockIdx.x + gridDim.x, ... of TP consecutive pixels of one image (the last tile of an image may
// be shorter), as (image, tile inside the image), without a 64-bit division per tile.  The producer and the consumers of a ring
// walk the same sequence: for (TileWalker t(hw, TP); t.image < n_img; t.next()).
struct TileWalker {
    int64_t tpi, image, tile_in_image;
    uint32_t step_images, step_tiles;
    MSPL_DEVINL TileWalker(int64_t hw, int tile_pix) : tpi((hw + tile_pix - 1) / tile_pix) {
        // blockIdx.x < gridDim.x < 2^31: a 32-bit division, with tiles per image beyond 32 bits clamped (same quotients)
        const uint32_t t = (uint32_t)(tpi < 0xffffffffll ? tpi : 0xffffffffll);
        image = blockIdx.x / t;
        tile_in_image = blockIdx.x % t;
        step_images = gridDim.x / t;
        step_tiles = gridDim.x % t;
    }
    MSPL_DEVINL void next() {
        image += step_images;
        tile_in_image += step_tiles;
        if (tile_in_image >= tpi) { tile_in_image -= tpi; ++image; }
    }
};

// the value of a run-time argument or of a std::integral_constant (whose conversion operator is host-only)
template <typename T> MSPL_DEVINL T cval(T v) { return v; }
template <typename T, T V> MSPL_DEVINL T cval(std::integral_constant<T, V>) { return V; }

// Body of listed shape SH (kSourceShapes): consume(ncls, seg, first) once per chunk, with the chunk's real class count, its
// group-end bits and whether it is the source's first chunk as compile-time constants.
template <int CH, int SH, typename Consume, int... I>
MSPL_DEVINL void consume_listed_shape(Consume& consume, std::integer_sequence<int, I...>) {
    constexpr SourceShape sh = kSourceShapes[SH];
    (consume(std::integral_constant<int, (sh.C - I * CH < CH ? sh.C - I * CH : CH)>{}, std::integral_constant<uint32_t, sh.seg[I]>{},
             std::bool_constant<I == 0>{}),
     ...);
}
// Runs the body of listed shape `shape` (ClassOrder::shape, 1-based); false when shape is 0 or not among SH + 1.
template <int CH, typename Consume, int... SH>
MSPL_DEVINL bool consume_listed_shapes(uint32_t shape, Consume& consume, std::integer_sequence<int, SH...>) {
    return ((shape == SH + 1 &&
             (consume_listed_shape<CH, SH>(consume, std::make_integer_sequence<int, kSourceShapes[SH].nchunk>{}), true)) ||
            ...);
}

// Producer warp of the full-resolution TMA kernels: walks this CTA's tiles in (tile, source, chunk) order and fills the ring.
// s_row: per-source class visiting order ([S][256] bytes in shared memory), or nullptr for the original class order.
// shaped: the consumers run the compiled bodies of listed shapes (ClassOrder::shape != 0), which never read the rows a tail
// chunk lacks, so those sources' tail chunks are not padded.
template <int NCW, int P, int CH, int NSTAGE>
MSPL_DEVINL void tma_produce_tiles(const FuseParams& prm, StageRing<NCW, NSTAGE>& ring, int lane, const uint8_t* s_row, bool shaped) {
    constexpr int TP = TmaCfg<NCW, P, CH, NSTAGE>::kTilePix;
    const int S = prm.S;
    const int64_t hw = prm.hw;
    const uint64_t policy = tma::evict_first_policy();
    for (TileWalker t(hw, TP); t.image < prm.n_img; t.next()) {
        const int64_t n = t.image;
        const int64_t off = t.tile_in_image * TP;
        const uint32_t row_bytes = (uint32_t)((hw - off < TP ? hw - off : TP) * sizeof(float));
        for (int s = 0; s < S; ++s) {
            const int C = prm.C[s];
            const float* pm = prm.main[s] + (n * C) * hw + off;
            const float* pa = prm.aux[s] + (n * C) * hw + off;
            const bool pad_tail = !(shaped && prm.order[s].shape != 0);
            for (int c0 = 0; c0 < C; c0 += CH) {
                const int cn = min(CH, C - c0);
                float* dst = ring.wait_empty();
                if (cn < CH && pad_tail) pad_tail_rows<CH>(dst, cn, lane, TP / 4, TP, CH * TP, TP / 4, TP);
                uint64_t* full = ring.expect(lane, 2 * cn * row_bytes);
                for (int j = lane; j < 2 * cn; j += 32) {
                    const int head = j >= cn, c = head ? j - cn : j;
                    const int cls = s_row ? (int)s_row[s * MSPL_MAX_SRC_CLASSES + c0 + c] : c0 + c;
                    const float* src = (head ? pa : pm) + (int64_t)cls * hw;
                    tma::bulk_g2s(dst + (head * CH + c) * TP, src, row_bytes, full, policy);
                }
                ring.advance();
            }
        }
    }
}

template <int NCW, int P, int CH, int NSTAGE, int KT, bool GK>
__global__ void __launch_bounds__((NCW + 1) * 32, 1) fuse_sources_tma_kernel(const __grid_constant__ FuseParams prm) {
    using Cfg = TmaCfg<NCW, P, CH, NSTAGE>;
    constexpr int TP = Cfg::kTilePix;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    StageRing<NCW, NSTAGE> ring(smem_raw, Cfg::kStageFloats);
    const TallySmem ts = tally_smem_init(prm, ring.end(), Cfg::kThreads, KT * Cfg::kThreads * P);
    ring.init();
    __syncthreads();

    const int S = prm.S;
    const int64_t hw = prm.hw;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    Tally<KT> tally;

    if (warp == NCW) {
        tma_produce_tiles<NCW, P, CH, NSTAGE>(prm, ring, lane, ts.row, CH == kFuseChunk);
    } else {
        // ------------------------------- consumer warps -------------------------------
        const float fS = 1.0f / (float)S;
        const int px = (warp * 32 + lane) * P;          // this thread's first pixel inside the tile
        Px<P>* group = reinterpret_cast<Px<P>*>(ts.group) + threadIdx.x;
        bool any_kld = false;
        for (int s = 0; s < S; ++s) any_kld |= prm.kld[s] != nullptr;
        for (TileWalker t(hw, TP); t.image < prm.n_img; t.next()) {
            const int64_t n = t.image;
            const int64_t off = t.tile_in_image * TP + px;
            const bool active = off < hw;                 // partial last tile: the ring holds stale values past the image
            PixelFusion<P, KT, GK> fus;
            fus.reset();
            for (int s = 0; s < S; ++s) {
                const int nchunk = (int)prm.order[s].nchunk;
                SourceStats<P> st;
                st.reset(group);
                // one chunk of ncls real classes: wait for its stage, copy the thread's values to registers, hand the stage
                // back, fold.  ncls is a compile-time count; seg and first are compile-time in the listed shapes' bodies.
                auto consume = [&](auto ncls, auto seg, auto first) {
                    constexpr int N = decltype(ncls)::value;
                    Px<P> m[CH], a[CH];
                    const float* src = ring.wait_full() + px;
#pragma unroll
                    for (int j = 0; j < N; ++j) m[j] = tma::lds_px<P>(src + j * TP);
#pragma unroll
                    for (int j = 0; j < N; ++j) a[j] = tma::lds_px<P>(src + (CH + j) * TP);
                    ring.release(lane);
                    fold_chunk<P, CH, N>(st, m, a, cval(first), cval(seg), Cfg::kThreads);
                };
                bool listed = false;
                if constexpr (CH == kFuseChunk)         // warp-uniform: one straight-line body per listed shape
                    listed = consume_listed_shapes<CH>(prm.order[s].shape, consume, std::make_integer_sequence<int, kNumSourceShapes>{});
                if (!listed) {
                    // Any other shape: the rescale runs on the first chunk's empty accumulators too (it evaluates to exact zeros,
                    // see SourceStats::reset), so the loop body is branch-free.  Measured and not kept: skipping it through a
                    // branch inside the loop (the merge costs ~20 register moves per chunk); peeling the first chunk out of the
                    // loop (4 MUFU and 11 packed operations less for 3 of the benchmark's 8 chunks per pixel pair, +1 % in bursts
                    // and nothing under the power limit); unrolling by 2 (164 instead of 171 instructions per chunk, 124
                    // registers).  Same bits in all of them.
                    using AllCH = std::integral_constant<int, CH>;
                    __builtin_assume(nchunk > 0);         // every source has a class: no zero-trip guard around the chunk loop
#pragma unroll 1
                    for (int chunk = 0; chunk < nchunk; ++chunk) consume(AllCH{}, prm.order[s].seg[chunk], false);
                }
                float d[P];
                fus.add_source(st, group, Cfg::kThreads, prm.order[s], d,
                               GlobalSlowPath<P>{prm, s, n, active ? off : 0, ts.lut + s * MSPL_MAX_SRC_CLASSES});
                if (any_kld) {     // per-source KLD maps are off in the label-generation job: one uniform test, hoisted
                    if (prm.kld[s] != nullptr && active) PixVec<P>::store(prm.kld[s] + n * hw + off, d);
                }
            }
            finish_tile(prm, fus, fS, tally, ts.hist, n, hw, off, active);
        }
    }
    tally.flush(prm, ts.hist, ts.cls, Cfg::kThreads);
}

// ----------------------------------------------------------------------------------------------------------------------
// Labels-only variant: what the reference's generation loop actually keeps (uest_seg_multi_os.py:900-921 discards the KLD and
// never forms a confidence).  With no confidence, uncertainty or histogram of confidences requested there is nothing to
// exponentiate: per class and pixel the consumers do z = m + a/2 and a running first-argmax (4 instructions), so the kernel
// is HBM-bound with a wide margin even at reduced clocks.  Same ring, same producer (original class order).
// ----------------------------------------------------------------------------------------------------------------------
template <int NCW, int P, int CH, int NSTAGE, int KT>
__global__ void __launch_bounds__((NCW + 1) * 32, 1) fuse_labels_tma_kernel(const __grid_constant__ FuseParams prm) {
    using Cfg = TmaCfg<NCW, P, CH, NSTAGE>;
    constexpr int TP = Cfg::kTilePix;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    StageRing<NCW, NSTAGE> ring(smem_raw, Cfg::kStageFloats);
    const TallySmem ts = tally_smem_init(prm, ring.end(), Cfg::kThreads);
    ring.init();
    __syncthreads();
    const int S = prm.S;
    const int64_t hw = prm.hw;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    Tally<KT> tally;
    if (warp == NCW) {
        tma_produce_tiles<NCW, P, CH, NSTAGE>(prm, ring, lane, nullptr, false);
    } else {
        const int px = (warp * 32 + lane) * P;
        for (TileWalker t(hw, TP); t.image < prm.n_img; t.next()) {
            const int64_t n = t.image;
            const int64_t off = t.tile_in_image * TP + px;
            const bool active = off < hw;
            uint32_t votes[P];
#pragma unroll
            for (int p = 0; p < P; ++p) votes[p] = 0;
            for (int s = 0; s < S; ++s) {
                const int C = prm.C[s];
                float best[P];
                int amax[P];
#pragma unroll
                for (int p = 0; p < P; ++p) { best[p] = -INFINITY; amax[p] = 0; }
#pragma unroll 1
                for (int c0 = 0; c0 < C; c0 += CH) {
                    float m[CH][P], a[CH][P];
                    const float* src = ring.wait_full() + px;
#pragma unroll
                    for (int j = 0; j < CH; ++j) tma::lds<P>(src + j * TP, m[j]);
#pragma unroll
                    for (int j = 0; j < CH; ++j) tma::lds<P>(src + (CH + j) * TP, a[j]);
                    ring.release(lane);
#pragma unroll
                    for (int j = 0; j < CH; ++j)
#pragma unroll
                        for (int p = 0; p < P; ++p) {
                            const float z = fmaf(0.5f, a[j][p], m[j][p]);     // as `pred + 0.5 * pred_aux` (:687); padded classes: -1.5e30
                            amax[p] = (z > best[p]) ? (c0 + j) : amax[p];    // strict >: first maximal index, as np.argmax (:904)
                            best[p] = fmaxf(best[p], z);
                        }
                }
#pragma unroll
                for (int p = 0; p < P; ++p) votes[p] += 1u << (4 * ts.lut[s * MSPL_MAX_SRC_CLASSES + amax[p]]);
            }
            int label[P];
            float conf[P];
            bool marg[P];
#pragma unroll
            for (int p = 0; p < P; ++p) {
                label[p] = merge_votes<KT>(votes[p], prm.vote_t, prm.ignore);
                conf[p] = 0.f;
                marg[p] = false;
            }
            if (active) store_labels<P>(prm.label + n * hw + off, label);
            tally.template add<P>(prm, ts.hist, label, conf, marg, off, active);
        }
    }
    tally.flush(prm, ts.hist, ts.cls, Cfg::kThreads);
}

// ======================================================================================================================
// K1-lowres: the same fusion, reading the sources' logits at their native (pre-upsample) resolution and performing the
// network's final bilinear align_corners=True interpolation in the consumer warps (next-row component, SURVEY.md 8f-1).
// HBM traffic drops from 8*sum(C) B/pixel to 4*sum(C)*(hm*wm + ha*wa)/(H*W) (1.25*sum(C) for the x2 / x4 heads of
// ESPDNetUE); the kernel is instruction-bound.
//   A tile is TP consecutive output pixels (row-major) of one image.  For every class of the chunk the producer copies
//   the block of source rows the tile's output rows interpolate from (whole rows, one bulk copy per class and head).
//   Source coordinates and weights follow ATen's upsample_bilinear2d (src = dst * (in-1)/(out-1); i = (int)src;
//   lambda = src - i); val = W00*v00 + W01*v01 + W10*v10 + W11*v11 (see PackedTaps), evaluated for the thread's two pixels at
//   once with packed multiplies / fmas: per class, head and PAIR of pixels 8 shared-memory loads + 4 packed instructions.
//   (A separable variant -- one warp-specialised vertical pass into a second shared-memory ring, then a 2-tap horizontal
//   pass per pixel -- was built and measured in round 2: 4.45 ms per 200 images with two blender warps against 2.08 ms
//   for the round-1 four-tap kernel; the vertical pass's address arithmetic and its extra hand-off cost more than the
//   taps it saves.  Not kept.)
//   MS / AS: compile-time class strides (floats) of the main / aux blocks inside a stage, or 0 to take them from the
//   geometry at run time.  With fixed strides every tap of every class is `LDS [tap_register + immediate]`.
// ======================================================================================================================
// Slow paths of K1-lowres: re-interpolate one pixel's logits from global memory with the fast path's own arithmetic.
static __device__ __noinline__ float lowres_logit_global(const float* __restrict__ src, int hin, int win, float rh, float rw, int y, int x) {
    const float hr = rh * (float)y, wr = rw * (float)x;
    const int i0 = (int)hr, x0 = (int)wr;
    const int dy = (i0 < hin - 1) ? win : 0, dx = (x0 < win - 1) ? 1 : 0;
    const float h1 = hr - (float)i0, h0 = 1.0f - h1;
    const float w1 = dx ? wr - (float)x0 : 0.0f, w0 = dx ? 1.0f - (wr - (float)x0) : 1.0f;      // as PackedTaps::set
    const float* p = src + (int64_t)i0 * win + x0;
    const float top = fmaf(w1, __ldg(p + dx), __fmul_rn(w0, __ldg(p))), bot = fmaf(w1, __ldg(p + dy + dx), __fmul_rn(w0, __ldg(p + dy)));
    return fmaf(h1, bot, __fmul_rn(h0, top));
}
template <int P>
struct LowresSlowPath {
    const float* gm;      // class 0 of image 0's main / aux head (the image's own is formed inside the rare branch)
    const float* ga;
    int64_t n;
    int C, hm, wm, ha, wa;
    float rhm, rwm, rha, rwa;
    int yy[P], xx[P];
    const uint8_t* lut;
    MSPL_DEVINL float z(int c, int p) const {
        return fmaf(0.5f, lowres_logit_global(ga + (n * C + c) * ha * wa, ha, wa, rha, rwa, yy[p], xx[p]),
                    lowres_logit_global(gm + (n * C + c) * hm * wm, hm, wm, rhm, rwm, yy[p], xx[p]));
    }
    MSPL_DEVINL float pmax(int p, float Mz) const {
        float s = 0.f;
#pragma unroll 1
        for (int c = 0; c < C; ++c) s += exp_neg(z(c, p) - Mz);
        return fminf(__frcp_rn(s), 1.0f);
    }
    MSPL_DEVINL int label(int p) const {
        float best = -INFINITY;
        int arg = 0;
#pragma unroll 1
        for (int c = 0; c < C; ++c) {
            const float v = z(c, p);
            if (v > best) { best = v; arg = c; }
        }
        return lut[arg];
    }
};

// One head's bilinear taps of a thread's P pixels inside a stage's class block (relative to the first staged source row).
// Only TWO offsets per pixel are kept -- the upper-left neighbour and the one below it (clamped at the last source row as ATen
// does) -- and the right-hand neighbours are read at +1 float through the load's immediate offset.  At the last source column
// ATen reads the same element twice (w1p = 0); here the horizontal weights are forced to (1, 0) there, so the +1 read (one float
// past the row: the next row, or finite slack inside the stage, which lowres_plan provides and the kernel zero-fills once) is
// multiplied by an exact zero.  Four registers of offsets instead of eight per head keeps the taps resident across the chunk
// loop -- with eight the compiler re-derived them from the pixel coordinates in every chunk (~70 instructions).
// The bilinear sample is evaluated as one chain over the four taps with the products of the vertical and horizontal weights
// formed once per tile, W00*v00 + W01*v01 + W10*v10 + W11*v11 (1 packed multiply + 3 packed fmas per class, head and pixel pair),
// not in ATen's nesting h0*(w0*v00 + w1*v01) + h1*(w0*v10 + w1*v11) (6 packed instructions).  The two differ in the last ulp of
// the interpolated logit, like the kernel and ATen do anyway (the parity definition of this row, DESIGN.md section 4, excuses
// exactly that); the kernel is bound by instruction issue, so the 20 instructions per chunk are worth ~5 %.
template <int P>
struct PackedTaps {
    int o0[P], o1[P];
    Px<P> w00, w01, w10, w11;
    MSPL_DEVINL void set(const int (&yy)[P], const int (&xx)[P], int hin, int win, float rh, float rw, int first_row) {
        float fw0[P], fw1[P], fh0[P], fh1[P];
#pragma unroll
        for (int p = 0; p < P; ++p) {
            const BilinearTap t = make_tap(yy[p], xx[p], hin, win, rh, rw, first_row);
            o0[p] = t.o00;
            o1[p] = t.o00 + t.dy;
            const bool last_col = t.dx == 0;
            fw0[p] = last_col ? 1.0f : t.w0; fw1[p] = last_col ? 0.0f : t.w1; fh0[p] = t.h0; fh1[p] = t.h1;
        }
        const Px<P> w0 = Px<P>::make(fw0), w1 = Px<P>::make(fw1), h0 = Px<P>::make(fh0), h1 = Px<P>::make(fh1);
        w00 = h0 * w0; w01 = h0 * w1; w10 = h1 * w0; w11 = h1 * w1;
    }
    template <int D>
    MSPL_DEVINL Px<P> gather(const float* __restrict__ s, const int (&o)[P]) const {
        float v[P];
#pragma unroll
        for (int p = 0; p < P; ++p) v[p] = s[o[p] + D];
        return Px<P>::make(v);
    }
    MSPL_DEVINL Px<P> interpolate(const float* __restrict__ s) const {
        Px<P> acc = w00 * gather<0>(s, o0);
        acc = fma(w01, gather<1>(s, o0), acc);
        acc = fma(w10, gather<0>(s, o1), acc);
        return fma(w11, gather<1>(s, o1), acc);
    }
};

template <int NCW, int P, int CH, int NSTAGE, int KT, bool GK, int MS = 0, int AS = 0>
__global__ void __launch_bounds__((NCW + 1) * 32, 1) fuse_sources_lowres_kernel(const __grid_constant__ FuseParams prm) {
    using Cfg = TmaCfg<NCW, P, CH, NSTAGE>;
    constexpr int kThreads = Cfg::kThreads;
    constexpr int TP = Cfg::kTilePix;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const LowresGeom& lr = prm.lr;
    const int main_stride = MS ? MS : lr.main_cls_stride, aux_stride = AS ? AS : lr.aux_cls_stride;
    const int aux_base = MS ? CH * MS : lr.aux_base;
    const int stage_floats = (MS && AS) ? CH * (MS + AS) : lr.stage_floats;
    StageRing<NCW, NSTAGE> ring(smem_raw, stage_floats);
    const TallySmem ts = tally_smem_init(prm, ring.end(), kThreads, KT * kThreads * P);
    // the +1-float reads of PackedTaps may touch floats no copy ever wrote (slack between class blocks): make them finite once
    for (int i = threadIdx.x; i < stage_floats * NSTAGE; i += kThreads) ring.base[i] = 0.f;
    ring.init();
    // generic-proxy writes above must be ordered before the async-proxy (bulk copy) writes into the same shared memory
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    __syncthreads();

    const int S = prm.S, H = lr.H, W = lr.W;
    const int64_t hw = prm.hw;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    Tally<KT> tally;

    if (warp == NCW) {
        // ------------------------------- producer warp -------------------------------
        const uint64_t policy = tma::evict_first_policy();
        for (TileWalker t(hw, TP); t.image < prm.n_img; t.next()) {
            const int64_t n = t.image;
            const int64_t off = t.tile_in_image * TP;
            const int y_first = (int)(off / W);
            const int64_t last = (off + TP < hw ? off + TP : hw) - 1;
            const int y_last = (int)(last / W);
            for (int s = 0; s < S; ++s) {
                const int C = prm.C[s], hm = lr.hm[s], wm = lr.wm[s], ha = lr.ha[s], wa = lr.wa[s];
                const float rhm = lowres_scale(hm, H), rha = lowres_scale(ha, H);
                const int m0 = (int)(rhm * (float)y_first), m1 = min((int)(rhm * (float)y_last) + 1, hm - 1);
                const int a0 = (int)(rha * (float)y_first), a1 = min((int)(rha * (float)y_last) + 1, ha - 1);
                const uint32_t mbytes = (uint32_t)((m1 - m0 + 1) * wm * sizeof(float));
                const uint32_t abytes = (uint32_t)((a1 - a0 + 1) * wa * sizeof(float));
                const float* pm = prm.main[s] + ((n * C) * hm + m0) * wm;
                const float* pa = prm.aux[s] + ((n * C) * ha + a0) * wa;
                for (int c0 = 0; c0 < C; c0 += CH) {
                    const int cn = min(CH, C - c0);
                    float* dst = ring.wait_empty();
                    if (cn < CH) pad_tail_rows<CH>(dst, cn, lane, (int)(mbytes / 16), main_stride, aux_base, (int)(abytes / 16), aux_stride);
                    uint64_t* full = ring.expect(lane, cn * (mbytes + abytes));
                    for (int j = lane; j < 2 * cn; j += 32) {
                        const int head = j >= cn, c = head ? j - cn : j;
                        const int cls = ts.row[s * MSPL_MAX_SRC_CLASSES + c0 + c];
                        if (head) tma::bulk_g2s(dst + aux_base + c * aux_stride, pa + (int64_t)cls * ha * wa, abytes, full, policy);
                        else tma::bulk_g2s(dst + c * main_stride, pm + (int64_t)cls * hm * wm, mbytes, full, policy);
                    }
                    ring.advance();
                }
            }
        }
    } else {
        // ------------------------------- consumer warps -------------------------------
        const float inv_s = 1.0f / (float)S;
        const int px = (warp * 32 + lane) * P;
        Px<P>* group = reinterpret_cast<Px<P>*>(ts.group) + threadIdx.x;
        for (TileWalker t(hw, TP); t.image < prm.n_img; t.next()) {
            const int64_t n = t.image;
            const int64_t tile_off = t.tile_in_image * TP;
            const int64_t off = tile_off + px;
            const bool active = off < hw;
            const int y_first = (int)(tile_off / W);
            int yy[P], xx[P];
#pragma unroll
            for (int p = 0; p < P; ++p) {
                const int64_t o = active ? off + p : tile_off;      // idle lanes interpolate the tile's first pixel
                yy[p] = (int)(o / W);
                xx[p] = (int)(o - (int64_t)yy[p] * W);
            }
            PixelFusion<P, KT, GK> fus;
            fus.reset();
            PackedTaps<P> tm, ta;
            for (int s = 0; s < S; ++s) {
                const int C = prm.C[s], hm = lr.hm[s], wm = lr.wm[s], ha = lr.ha[s], wa = lr.wa[s];
                const float rhm = lowres_scale(hm, H), rwm = lowres_scale(wm, W);
                const float rha = lowres_scale(ha, H), rwa = lowres_scale(wa, W);
                if (s == 0 || !lr.same_geometry) {      // sources of one architecture share their head sizes: taps once per tile
                    tm.set(yy, xx, hm, wm, rhm, rwm, (int)(rhm * (float)y_first));
                    ta.set(yy, xx, ha, wa, rha, rwa, (int)(rha * (float)y_first));
                }
                SourceStats<P> st;
                st.reset(group);
                const int nchunk = (int)prm.order[s].nchunk;
                __builtin_assume(nchunk > 0);
                auto consume = [&](int chunk, bool first) {
                    Px<P> m[CH], a[CH];
                    const float* src = ring.wait_full();
#pragma unroll
                    for (int j = 0; j < CH; ++j) {
                        m[j] = tm.interpolate(src + j * main_stride);
                        a[j] = ta.interpolate(src + aux_base + j * aux_stride);
                    }
                    ring.release(lane);
                    fold_chunk<P, CH>(st, m, a, first, prm.order[s].seg[chunk], kThreads);
                };
                // The first chunk is peeled out of the loop as a straight-line copy of the body without the rescale of the empty
                // accumulators.  This kernel is bound by instruction issue, not by HBM or board power, so that is worth 4.5 %
                // here (1.895 -> 1.810 ms per 200 images, same-box A/B, identical outputs).  Unrolling the loop by 2 removes its
                // loop-carried register moves but measured +1.7 % time without GK (it spills there) and -0.4 % with GK (1.797
                // -> 1.790 ms per 200 images): not worth the code size.
                consume(0, true);
#pragma unroll 1
                for (int chunk = 1; chunk < nchunk; ++chunk) consume(chunk, false);
                float d[P];
                LowresSlowPath<P> slow{prm.main[s], prm.aux[s], n, C, hm, wm, ha, wa,
                                       rhm, rwm, rha, rwa, {}, {}, ts.lut + s * MSPL_MAX_SRC_CLASSES};
#pragma unroll
                for (int p = 0; p < P; ++p) { slow.yy[p] = yy[p]; slow.xx[p] = xx[p]; }
                fus.add_source(st, group, kThreads, prm.order[s], d, slow);
                if (prm.kld[s] != nullptr && active) PixVec<P>::store(prm.kld[s] + n * hw + off, d);
            }
            finish_tile(prm, fus, inv_s, tally, ts.hist, n, hw, off, active);
        }
    }
    tally.flush(prm, ts.hist, ts.cls, kThreads);
}

}  // namespace mspl
