// Per-pixel statistics of one source's (main, aux) logit pair, accumulated chunk by chunk.
//
// For a pixel with class logits m_c (main head) and a_c (aux head), z_c = m_c + 0.5*a_c, the reference needs
//   softmax(z)                  uest_seg_multi_os.py:687-689
//   first-argmax_c -> LUT       uest_seg_multi_os.py:904-912  (decided on z: softmax is monotone; ties -> lowest c)
//   KL(softmax(m)||softmax(a))  loss_fns/segmentation_loss.py:181-189
// All of them follow from the running quantities below, updated one chunk of CH classes at a time (online
// softmax: a chunk's maxima are folded in with ONE rescale per chunk, not one per class):
//   Mm, Sm = sum e^{m-Mm}     Ma, Sa = sum e^{a-Ma}     Sz = sum e^{z-Rz}     T = sum e^{m-Mm} ((m-Mm) - (a-Ma))
//   g_k = max z over the source classes the label table maps to target class k
// Then  KLD = T/Sm - log Sm + log Sa   (the reference's sum_c p1*(logp1 - logp2), with log_softmax written as
// (x - max) - log(sum) exactly as ATen does, so no large maxima are ever added back),
// Mz = max_k g_k, label = the k attaining it, max prob = e^{Mz-Rz}/Sz, G_s[k] = e^{g_k-Rz}/Sz.
//
// Two things keep the instruction count per class and pixel low (the kernels are co-limited by issue slots):
//   * a thread's P = 2 neighbouring pixels travel as ONE 64-bit register pair and every add / multiply / fma on them is a
//     packed Blackwell instruction (FADD2 / FMUL2 / FFMA2: two fp32 lanes per issue slot, IEEE results identical to the
//     scalar forms); only the maxima and the MUFU exponentials are issued per lane;
//   * the classes of a source are visited GROUPED BY TARGET CLASS (the loaders fetch class rows in that order, see
//     ClassOrder): no arg-max index is tracked, only a running maximum of z that is committed to its target's slot at the
//     (warp-uniform) group boundaries.  The reference's first-maximal-index rule only matters when two DIFFERENT targets tie
//     exactly; that is detected from the committed maxima and resolved out of line in the original class order.
#pragma once
#include "common.cuh"

namespace mspl {

// e^t for t <= 0 (t already max-subtracted, so the largest term is exactly e^0 = 1): FMUL + MUFU.EX2.
MSPL_DEVINL float ex2_approx(float x) {
    float r;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}
MSPL_DEVINL float exp_neg(float t) { return ex2_approx(t * kLog2e); }
MSPL_DEVINL float exp_half_neg(float t) { return ex2_approx(t * (0.5f * kLog2e)); }   // e^{t/2}
// natural log through MUFU.LG2 (absolute error <= 2^-22.6 * |log2 x| * ln 2: ~5e-7 at worst for the ratios of softmax sums it
// is used on, inside the 2e-6 KLD floor), instead of the ~20-instruction branchy logf
MSPL_DEVINL float lg2_approx(float x) {
    float r;
    asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}
constexpr float kLn2 = 0.6931471805599453f;
MSPL_DEVINL float log_fast(float x) { return lg2_approx(x) * kLn2; }
// 1/x through MUFU.RCP alone (relative error <= 2^-23; the IEEE sequence adds a Newton step and a range check per call)
MSPL_DEVINL float rcp_fast(float x) {
    float r;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}
MSPL_DEVINL float max3(float a, float b, float c) {        // FMNMX3 (sm_100+)
    float r;
    asm("max.f32 %0, %1, %2, %3;" : "=f"(r) : "f"(a), "f"(b), "f"(c));
    return r;
}

// ---- P pixels of one thread as one value ------------------------------------------------------------------------------
// Px<2>: two fp32 lanes in one 64-bit register pair, arithmetic through the packed f32x2 instructions (sm_100+).
// Px<1>: plain float (the scalar fallback kernel for unaligned shapes).  Same IEEE results lane for lane.
template <int P> struct Px;

template <> struct Px<1> {
    float v;
    static MSPL_DEVINL Px splat(float x) { return Px{x}; }
    static MSPL_DEVINL Px make(const float (&a)[1]) { return Px{a[0]}; }
    MSPL_DEVINL void get(float (&a)[1]) const { a[0] = v; }
    // load from shared memory HERE (a volatile access keeps its place: the compiler would otherwise sink it into a later branch)
    static MSPL_DEVINL Px load_shared_now(const Px* p) {
        Px r;
        asm volatile("ld.volatile.shared.f32 %0, [%1];" : "=f"(r.v) : "r"((uint32_t)__cvta_generic_to_shared(p)));
        return r;
    }
};
// (the _rn intrinsics are never contracted into fused multiply-adds, so the scalar kernel rounds exactly where the packed
//  instructions do and both produce the same bits)
MSPL_DEVINL Px<1> operator+(Px<1> a, Px<1> b) { return Px<1>{__fadd_rn(a.v, b.v)}; }
MSPL_DEVINL Px<1> operator-(Px<1> a, Px<1> b) { return Px<1>{__fsub_rn(a.v, b.v)}; }
MSPL_DEVINL Px<1> operator*(Px<1> a, Px<1> b) { return Px<1>{__fmul_rn(a.v, b.v)}; }
MSPL_DEVINL Px<1> fma(Px<1> a, Px<1> b, Px<1> c) { return Px<1>{fmaf(a.v, b.v, c.v)}; }

template <> struct Px<2> {
    unsigned long long v;
    static MSPL_DEVINL Px pack(float lo, float hi) {
        Px r;
        asm("mov.b64 %0, {%1, %2};" : "=l"(r.v) : "f"(lo), "f"(hi));
        return r;
    }
    static MSPL_DEVINL Px splat(float x) { return pack(x, x); }
    static MSPL_DEVINL Px make(const float (&a)[2]) { return pack(a[0], a[1]); }
    MSPL_DEVINL void get(float (&a)[2]) const { asm("mov.b64 {%0, %1}, %2;" : "=f"(a[0]), "=f"(a[1]) : "l"(v)); }
    static MSPL_DEVINL Px load_shared_now(const Px* p) {
        Px r;
        asm volatile("ld.volatile.shared.b64 %0, [%1];" : "=l"(r.v) : "r"((uint32_t)__cvta_generic_to_shared(p)));
        return r;
    }
};
MSPL_DEVINL Px<2> operator+(Px<2> a, Px<2> b) {
    Px<2> r;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r.v) : "l"(a.v), "l"(b.v));
    return r;
}
MSPL_DEVINL Px<2> operator-(Px<2> a, Px<2> b) {
    Px<2> r;
    asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(r.v) : "l"(a.v), "l"(b.v));
    return r;
}
MSPL_DEVINL Px<2> operator*(Px<2> a, Px<2> b) {
    Px<2> r;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r.v) : "l"(a.v), "l"(b.v));
    return r;
}
MSPL_DEVINL Px<2> fma(Px<2> a, Px<2> b, Px<2> c) {
    Px<2> r;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r.v) : "l"(a.v), "l"(b.v), "l"(c.v));
    return r;
}

// lane-wise helpers (issued per lane: there is no packed FMNMX / MUFU)
template <int P, typename F>
MSPL_DEVINL Px<P> lanewise(Px<P> a, F f) {
    float x[P];
    a.get(x);
#pragma unroll
    for (int p = 0; p < P; ++p) x[p] = f(x[p]);
    return Px<P>::make(x);
}
template <int P>
MSPL_DEVINL Px<P> pmax(Px<P> a, Px<P> b) {
    float x[P], y[P];
    a.get(x); b.get(y);
#pragma unroll
    for (int p = 0; p < P; ++p) x[p] = fmaxf(x[p], y[p]);
    return Px<P>::make(x);
}
template <int P>
MSPL_DEVINL Px<P> pmin(Px<P> a, Px<P> b) {
    float x[P], y[P];
    a.get(x); b.get(y);
#pragma unroll
    for (int p = 0; p < P; ++p) x[p] = fminf(x[p], y[p]);
    return Px<P>::make(x);
}
template <int P>
MSPL_DEVINL Px<P> pmax3(Px<P> a, Px<P> b, Px<P> c) {
    float x[P], y[P], z[P];
    a.get(x); b.get(y); c.get(z);
#pragma unroll
    for (int p = 0; p < P; ++p) x[p] = max3(x[p], y[p], z[p]);
    return Px<P>::make(x);
}
// max of init and the first N entries of v
template <int P, int N, int L>
MSPL_DEVINL Px<P> pmax_of(const Px<P> (&v)[L], Px<P> init) {
    static_assert(N <= L, "pmax_of reads past the array");
    Px<P> r = init;
    int j = 0;
#pragma unroll
    for (; j + 1 < N; j += 2) r = pmax3<P>(r, v[j], v[j + 1]);
    if (j < N) r = pmax<P>(r, v[j]);
    return r;
}
template <int P> MSPL_DEVINL Px<P> pex2(Px<P> a) { return lanewise<P>(a, [](float x) { return ex2_approx(x); }); }

// ---- class visiting order of one source -----------------------------------------------------------------------------
// Built on the host from the label table (build_class_order in fuse_launch.cuh): row[i] = the source class fetched i-th,
// classes sorted by (target class, class index).  seg[chunk]: bit j = slot j of the chunk is the LAST class of its target
// group.  `present` = bit k set when some class maps to target k; the groups are committed in ascending k, so the i-th
// committed maximum belongs to the i-th set bit of `present`.
constexpr int kMaxChunksPerSource = 64;       // >= ceil(MSPL_MAX_SRC_CLASSES / CH) for every CH >= 4
struct ClassOrder {
    uint8_t row[MSPL_MAX_SRC_CLASSES];
    uint8_t seg[kMaxChunksPerSource];
    uint32_t present;
    uint32_t nchunk;          // ceil(C / CH) for the chunk size the order was built for
    uint32_t ngroup;          // number of target groups = popcount(present) (>= 1)
    uint32_t vote[MSPL_MAX_CLASSES];   // vote[i] = 1 << 4*(target class of the i-th committed group): what a source adds to a
                                       // pixel's packed vote counters (4 bits per target) when group i holds its largest z
    uint32_t shape;           // 1 + index into kSourceShapes when (C, nchunk, seg) is a listed shape, else 0
};

// ---- compiled chunk shapes ---------------------------------------------------------------------------------------------
// Everything the chunk loop does per source follows from (C, nchunk, seg[0..nchunk)) alone.  The shapes of the greenhouse
// tables (data_loader/segmentation/greenhouse.py SOURCE_TABLES, at kFuseChunk classes per chunk) are listed here, and the
// TMA kernel runs a fully unrolled body for each of them: group commits only where a group ends, no rescale on the first chunk,
// and a tail chunk that loads and folds only its real classes (so the producer writes no padding for it).  Any other shape
// runs the generic loop.  build_class_order sets ClassOrder::shape.
// kFuseChunk is the chunk size of every K1 kernel the library launches (classes per chunk: 13 -> 5+5+3, 20 -> 4x5, 5 -> one
// exact two-sweep chunk, picked from the tools/k1_sweep measurements on B200, see profiles/).
constexpr int kFuseChunk = 5;
constexpr int kMaxShapeChunks = 4;
struct SourceShape {
    int C, nchunk;
    uint8_t seg[kMaxShapeChunks];
};
constexpr SourceShape kSourceShapes[] = {
    {13, 3, {0x01, 0x0a, 0x04}},          // camvid: groups of 1, 6, 2, 4 classes
    {20, 4, {0x01, 0x00, 0x04, 0x11}},    // cityscapes: 1, 12, 3, 4
    {5, 1, {0x1a}},                       // forest: 2, 2, 1
};
constexpr int kNumSourceShapes = (int)(sizeof(kSourceShapes) / sizeof(kSourceShapes[0]));

// Running per-pixel statistics of one source.
//   Mm, Sm = sum e^{m-Mm}     Ma, Sa = sum e^{a-Ma}     T = sum e^{m-Mm} ((m-Mm) - (a-Ma))
//   Sz = sum e^{z - Rz} with the reference point Rz = Mm + Ma/2 (>= max z): e^{z-Rz} = e^{m-Mm} * e^{(a-Ma)/2}, so the
//        z-softmax costs no exponential of its own (two MUFU.EX2 per class instead of three).
//   run = max z over the classes of the target group being visited (committed to the group's slot at its last class)
//   slot = where the next finished group's maximum goes: the groups of a source are committed in visiting order (ascending
//          target class) to consecutive entries of the thread's column, `gstride` apart
template <int P>
struct SourceStats {
    Px<P> Mm, Sm, Ma, Sa, Sz, T, run;
    Px<P>* slot;
    MSPL_DEVINL void reset(Px<P>* group) {
        // finite sentinel (not -inf) for the softmax maxima: the rescale of an empty accumulator then evaluates to exactly 0
        // without NaNs, so kernels may run it unconditionally on a source's first chunk
        Mm = Ma = Px<P>::splat(-1.0e30f);
        Sm = Sa = Sz = T = Px<P>::splat(0.f);
        run = Px<P>::splat(-INFINITY);
        slot = group;
    }
};

// Value loaded in place of the classes a tail chunk does not have: hugely negative but finite, so that it never wins a
// max, its exponentials are exactly 0 and (m - Mm) - (a - Ma) stays finite (0) -- the math below needs no predicates.
constexpr float kPadLogit = -1.0e30f;

// Fold the first N (default CH) classes of one chunk into the running stats.  m/a hold the chunk's logits in visiting order;
// with N = CH, entries past the source's last class are kPadLogit; entries from N on are not read.  The rescale of a first
// chunk adds exact zeros, and so do padded classes once any logit of the source lies above kPadLogit: N = the real class
// count and N = CH with padding give the same bits, and so does either `first` on a first chunk.
// `first` (warp-uniform): nothing accumulated yet, skip the rescale.  seg: the chunk's ClassOrder word (bit j: slot j ends
// its target group).  Finished groups go to st.slot, gstride entries apart.
template <int P, int CH, int N = CH>
MSPL_DEVINL void fold_chunk(SourceStats<P>& st, const Px<P> (&m)[CH], const Px<P> (&a)[CH], bool first, uint32_t seg, int gstride) {
    static_assert(0 < N && N <= CH, "a chunk folds 1..CH classes");
    const Px<P> half = Px<P>::splat(0.5f);
    // sweep 1: z exactly as the reference forms it (0.5*a is exact in fp32, so the fused multiply-add rounds once, just
    // like `pred + 0.5 * pred_aux`), folded into the running maximum of the current target group
#pragma unroll
    for (int j = 0; j < N; ++j) {
        st.run = pmax<P>(st.run, fma(a[j], half, m[j]));
        if ((seg >> j) & 1u) {              // warp-uniform: last class of its group
            *st.slot = st.run;
            st.slot += gstride;
            st.run = Px<P>::splat(-INFINITY);
        }
    }
    const Px<P> nMm = pmax_of<P, N>(m, st.Mm), nMa = pmax_of<P, N>(a, st.Ma);
    Px<P> sm_old = Px<P>::splat(0.f), rm = sm_old, sm, sa = sm_old, sz = sm_old, t = sm_old;
    const Px<P> l2e = Px<P>::splat(kLog2e), hl2e = Px<P>::splat(0.5f * kLog2e);
    if (!first) {   // rescale what earlier chunks accumulated to the new maxima
        const Px<P> dm = st.Mm - nMm, da = st.Ma - nMa;
        const Px<P> rh = pex2<P>(da * hl2e);
        rm = pex2<P>(dm * l2e);
        sm_old = st.Sm;
        t = rm * fma(st.Sm, dm - da, st.T);
        sa = st.Sa * (rh * rh);
        sz = st.Sz * (rm * rh);
    }
    // sweep 2: the exponentials and the four sums.  The rescaled old sum Sm*rm enters through an EXPLICIT fma with the first
    // class's term: ptxas fuses a packed multiply into a following packed add whenever it sees the pair, so spelling it out
    // keeps every variant of the kernels (packed / scalar, with / without the first-chunk branch) on the same bits.
#pragma unroll
    for (int j = 0; j < N; ++j) {
        const Px<P> tm = m[j] - nMm, ta = a[j] - nMa;
        const Px<P> em = pex2<P>(tm * l2e), h = pex2<P>(ta * hl2e);
        sm = (j == 0) ? fma(sm_old, rm, em) : sm + em;
        t = fma(em, tm - ta, t);
        sa = fma(h, h, sa);
        sz = fma(em, h, sz);
    }
    st.Mm = nMm; st.Ma = nMa;
    st.Sm = sm; st.Sa = sa; st.Sz = sz; st.T = t;
}

// What the fusion needs from a finished source, for the thread's P pixels at once (packed like the running statistics: the
// adds / multiplies are one instruction for both pixels, only MUFU and min/max are issued per lane).
template <int P>
struct SourceResult {
    Px<P> kld;      // KL(softmax(m) || softmax(a)) = T/Sm - log Sm + log Sa  (= sum_c p1 (logp1 - logp2), log_softmax taken as
                    // (x - max) - log(sum) like ATen, so no large maxima are ever added back)
    Px<P> rz;       // Rz = Mm + Ma/2, the reference point of Sz
    Px<P> inv_sz;   // 1 / Sz:  softmax(z)_c = e^{z_c - Rz} * inv_sz
    Px<P> pmax;     // probability of the argmax class = e^{Mz - Rz} * inv_sz
    Px<P> gap;      // Mz - Rz (<= 0): the caller's degeneracy test reads it
};

// Largest Rz - Mz for which the shared exponentials are trusted.  e^{z-Rz} is formed as a product of two MUFU.EX2 results
// whose arguments grow with the gap; an argument of magnitude 2^e carries an absolute rounding error of 2^(e-24), i.e. a
// relative error of ~0.7 * 2^(e-24) in the exponential.  Up to a gap of 16 (arguments < 32) the confidence stays within
// ~3e-6 of the exact softmax; at 64 -- where Sz would start to underflow -- it would be 3e-5 (seen by the seeded sweep in
// tests/test_gpu_fuzz.py on logits of standard deviation 40).  Network logits are O(10): the slow path is never taken on
// the benchmark's inputs, it exists so that pathological inputs still meet the 1e-5 tolerance.
constexpr float kMaxSharedExpGap = 16.f;
// Largest |Mz| for the same.  The reference takes the softmax of z AFTER rounding it to fp32 (`pred + 0.5*pred_aux`), the
// shared exponentials work on the unrounded sum (m-Mm) + (a-Ma)/2 and on a separately rounded Rz: the two differ by up to
// ~1.5 ulp(z) in the exponent: at most 7.6e-6 relative up to |Mz| = 48 (|Rz| <= 64), but 3e-5 at |z| = 256.  Beyond 48 the
// slow path recomputes the reference's own expression e^{z_c - Mz} from the rounded z.  (A limit of 32 put ~3 pixels in 10^5
// of the benchmark's N(0, 6.4^2) fused logits on the slow path and cost K1 1.6 %; 48 is 7.5 sigma away.)
constexpr float kMaxSharedExpLogit = 48.f;

// Mz: the maximum of the source's fused logits, per pixel.
template <int P>
MSPL_DEVINL SourceResult<P> finish_source(const SourceStats<P>& st, Px<P> Mz) {
    SourceResult<P> r;
    const Px<P> inv_sm = lanewise<P>(st.Sm, [](float x) { return rcp_fast(x); });
    const Px<P> lg2 = lanewise<P>(st.Sa * inv_sm, [](float x) { return lg2_approx(x); });
    r.kld = fma(st.T, inv_sm, lg2 * Px<P>::splat(kLn2));
    r.rz = fma(Px<P>::splat(0.5f), st.Ma, st.Mm);
    r.inv_sz = lanewise<P>(st.Sz, [](float x) { return rcp_fast(x); });
    r.gap = Mz - r.rz;
    // numerator and its term of Sz round separately: clamp
    r.pmax = pmin<P>(pex2<P>(r.gap * Px<P>::splat(kLog2e)) * r.inv_sz, Px<P>::splat(1.0f));
    return r;
}
// the two heads' maxima sit more than kMaxSharedExpGap logit units above Mz, or |Mz| is beyond the trusted range: the caller
// takes the slow path for this pixel (also catches NaN)
MSPL_DEVINL bool degenerate_source(float gap, float Mz) { return !(gap >= -kMaxSharedExpGap) || !(fabsf(Mz) <= kMaxSharedExpLogit); }

// ---- out-of-line slow paths (rare, divergent): they must not bloat the hot loop's instruction footprint ----------------
// Degenerate pixel: recompute 1/sum_c e^{z_c - Mz} directly from global memory.
static __device__ __noinline__ float recompute_pmax(const float* __restrict__ pm, const float* __restrict__ pa, int C, int64_t hw, float Mz) {
    float s = 0.f;
#pragma unroll 1
    for (int c = 0; c < C; ++c) s += exp_neg(fmaf(0.5f, __ldg(pa + c * hw), __ldg(pm + c * hw)) - Mz);
    return __frcp_rn(s);
}
// Two different target classes tie exactly for the maximum of z: the reference's label is the table entry of the FIRST maximal
// class in the original class order (np.argmax, uest_seg_multi_os.py:904).
static __device__ __noinline__ int recompute_label(const float* __restrict__ pm, const float* __restrict__ pa, int C, int64_t hw,
                                                   const uint8_t* lut) {
    float best = -INFINITY;
    int arg = 0;
#pragma unroll 1
    for (int c = 0; c < C; ++c) {
        const float z = fmaf(0.5f, __ldg(pa + c * hw), __ldg(pm + c * hw));
        if (z > best) { best = z; arg = c; }       // strict >: lowest index wins ties
    }
    return lut[arg];
}

}  // namespace mspl
