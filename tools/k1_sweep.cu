// tools/k1_sweep -- times variants of the fused K1 kernel (direct-load and TMA-staged) on synthetic logits.
// Development tool, not part of the library: prints one line per variant with ms, algorithmic GB/s (313 B/pixel for the
// 13/20/5-class configuration) and a checksum of the outputs so that variants can be compared for equality.
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "../mspl_b200/csrc/fuse_launch.cuh"

using namespace mspl;

__global__ void fill_logits(float* main_l, float* aux_l, int64_t n, uint32_t seed, int C, int64_t hw) {
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        uint32_t x = (uint32_t)(i * 2654435761u) ^ seed;
        float acc = 0.f, acc2 = 0.f;
        for (int r = 0; r < 4; ++r) {          // sum of uniforms ~ normal
            x ^= x << 13; x ^= x >> 17; x ^= x << 5;
            acc += (x & 0xffff) * (1.0f / 65536.0f) - 0.5f;
            acc2 += (x >> 16) * (1.0f / 65536.0f) - 0.5f;
        }
        const int c = (int)((i / hw) % C);
        const float m = 3.0f * 1.7320508f * acc + 1.5f * ((c * 7 + 3) % 5 - 2);   // class bias -> non-uniform labels
        main_l[i] = m;
        aux_l[i] = m + 1.5f * 1.7320508f * acc2;
    }
}

__global__ void checksum_kernel(const uint8_t* label, const float* conf, const float* unc, int64_t n, unsigned long long* out) {
    unsigned long long a = 0, b = 0, c = 0;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        a += label[i] * (unsigned long long)((i % 1021) + 1);
        b += __float_as_uint(conf[i]) >> 8;
        c += __float_as_uint(unc[i]) >> 12;
    }
    atomicAdd(out, a); atomicAdd(out + 1, b); atomicAdd(out + 2, c);
}

struct Bench {
    FuseParams prm;
    int64_t npix;
    unsigned long long* d_stats;   // class_hist[8], marginal, conf_hist[8*2048], checksum[3]
    int reps;
    float soak_s = 0.f;
};

template <typename F>
static void run_variant(const char* name, Bench& b, F launch) {
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0); cudaEventCreate(&e1);
    const size_t stats_bytes = sizeof(unsigned long long) * (8 + 8 + 8 * 2048 + 8);
    cudaMemset(b.d_stats, 0, stats_bytes);
    int rc = launch();
    cudaError_t err = cudaDeviceSynchronize();
    if (rc != 0 || err != cudaSuccess) {
        printf("%-44s FAILED rc=%d cuda=%s\n", name, rc, cudaGetErrorString(err));
        cudaGetLastError();
        return;
    }
    unsigned long long h[16];
    checksum_kernel<<<592, 256>>>(b.prm.label, b.prm.conf, b.prm.unc, b.npix, b.d_stats + 16 + 8 * 2048);
    cudaMemcpy(h, b.d_stats, sizeof(unsigned long long) * 16, cudaMemcpyDeviceToHost);
    unsigned long long cs[3];
    cudaMemcpy(cs, b.d_stats + 16 + 8 * 2048, sizeof(cs), cudaMemcpyDeviceToHost);
    launch();
    if (b.soak_s > 0.f) {      // keep the board under load first, so that a power limiter (if this box has one that bites) has settled
        cudaEventRecord(e0);
        float el = 0.f;
        while (el < b.soak_s * 1e3f) {
            for (int i = 0; i < 8; ++i) launch();
            cudaEventRecord(e1);
            cudaEventSynchronize(e1);
            cudaEventElapsedTime(&el, e0, e1);
        }
    }
    float best = 1e30f, sum = 0.f;
    for (int r = 0; r < b.reps; ++r) {
        cudaEventRecord(e0);
        launch();
        cudaEventRecord(e1);
        cudaEventSynchronize(e1);
        float ms;
        cudaEventElapsedTime(&ms, e0, e1);
        best = ms < best ? ms : best;
        sum += ms;
    }
    const double bytes = (double)b.npix * 313.0;
    printf("%-44s min %8.3f ms  mean %8.3f ms  %7.1f GB/s (min)  frac6455 %.3f  | hist %llu %llu %llu %llu %llu marg %llu cs %llx %llx %llx\n", name, best,
           sum / b.reps, bytes / 1e6 / best, bytes / 1e6 / best / 6455.6, h[0], h[1], h[2], h[3], h[4], h[8], cs[0], cs[1], cs[2]);
    fflush(stdout);
    if (b.soak_s > 0.f) {
        for (int i = 0; i < 4; ++i) launch();      // still busy while nvidia-smi samples
        if (system("nvidia-smi -i 0 --query-gpu=clocks.sm,clocks.mem,power.draw,clocks_event_reasons.sw_power_cap --format=csv,noheader | sed 's/^/    clocks under load: /'") != 0) {}
        cudaDeviceSynchronize();
    }
    cudaEventDestroy(e0); cudaEventDestroy(e1);
}

#define DIRECT(CH, THREADS, MINB, GK)                                                                                            \
    if (want(#CH "," #THREADS "," #MINB, "direct")) {                                                                            \
        build_class_order(b.prm, CH);                                                                                            \
        run_variant("direct P=1 CH=" #CH " thr=" #THREADS " minb=" #MINB " gk=" #GK, b, [&] {                                  \
            return launch_fuse_direct<THREADS>(fuse_sources_direct_kernel<CH, 5, GK, THREADS, MINB>, b.prm, 5, 0);               \
        });                                                                                                                      \
    }
#define TMA(NCW, P, CH, NST, GK)                                                                                                 \
    if (want(#NCW "," #P "," #CH "," #NST, "tma")) {                                                                             \
        using Cfg = TmaCfg<NCW, P, CH, NST>;                                                                                     \
        build_class_order(b.prm, CH);                                                                                            \
        if (tma_eligible(b.prm) && Cfg::smem_bytes(5, 5) <= 227 * 1024)                                                          \
            run_variant("tma ncw=" #NCW " P=" #P " CH=" #CH " stages=" #NST " gk=" #GK, b, [&] {                               \
                return launch_fuse_ring<Cfg>(fuse_sources_tma_kernel<NCW, P, CH, NST, 5, GK>, b.prm, Cfg::smem_bytes(5, 5), 0); \
            });                                                                                                                  \
        else printf("tma ncw=" #NCW " P=" #P " CH=" #CH " stages=" #NST ": not eligible / smem %zu\n", Cfg::smem_bytes(5, 5));  \
    }

#define LABELS(NCW, P, CH, NST)                                                                                                  \
    if (want(#NCW "," #P "," #CH "," #NST, "labels")) {                                                                          \
        using Cfg = TmaCfg<NCW, P, CH, NST>;                                                                                     \
        FuseParams q = b.prm;                                                                                                    \
        q.conf = nullptr; q.unc = nullptr; q.conf_hist = nullptr; q.marginal = nullptr;                                         \
        build_class_order(q, CH);                                                                                                \
        run_variant("labels-only ncw=" #NCW " P=" #P " CH=" #CH " stages=" #NST " (no softmax: z, arg-max, table, vote)", b, [&] { \
            return launch_fuse_ring<Cfg>(fuse_labels_tma_kernel<NCW, P, CH, NST, 5>, q, Cfg::smem_bytes(5, 5), 0);              \
        });                                                                                                                      \
    }

#define LOWRES(NCW, P, CH, NST, GK)                                                                                              \
    if (want(#NCW "," #P "," #NST, "lowres")) {                                                                                  \
        FuseParams q = b.prm;                                                                                                    \
        build_class_order(q, CH);                                                                                                \
        const size_t smem = lowres_plan(q, NCW * 32 * P, CH, NST, 5, (NCW + 1) * 32, P, 768, 384);                               \
        if (smem && smem <= 227 * 1024)                                                                                          \
            run_variant("lowres ncw=" #NCW " P=" #P " CH=" #CH " stages=" #NST " gk=" #GK, b, [&] {                            \
                return launch_fuse_ring<TmaCfg<NCW, P, CH, NST>>(fuse_sources_lowres_kernel<NCW, P, CH, NST, 5, GK, 768, 384>, q, \
                                                                 smem, 0);                                               \
            });                                                                                                                  \
        else printf("lowres ncw=" #NCW " stages=" #NST ": smem %zu does not fit\n", smem);                                     \
    }

static const char* g_filter = nullptr;
static bool want(const char* key, const char* family) {
    if (!g_filter) return true;
    return strstr(g_filter, family) != nullptr || strstr(g_filter, key) != nullptr;
}

int main(int argc, char** argv) {
    int64_t n_img = 400, H = 256, W = 480;
    int reps = 5, vote_t = 3, policy = MSPL_POLICY_VOTE;
    bool hist = true, lowres = false;
    float soak = 0.f;
    for (int i = 1; i < argc; ++i) {
        if (!strcmp(argv[i], "--images")) n_img = atoll(argv[++i]);
        else if (!strcmp(argv[i], "--reps")) reps = atoi(argv[++i]);
        else if (!strcmp(argv[i], "--hw")) { H = atoll(argv[++i]); W = atoll(argv[++i]); }
        else if (!strcmp(argv[i], "--vote")) vote_t = atoi(argv[++i]);
        else if (!strcmp(argv[i], "--prob")) policy = MSPL_POLICY_PROB;
        else if (!strcmp(argv[i], "--nohist")) hist = false;
        else if (!strcmp(argv[i], "--lowres")) lowres = true;
        else if (!strcmp(argv[i], "--only")) g_filter = argv[++i];
        else if (!strcmp(argv[i], "--soak")) soak = (float)atof(argv[++i]);
    }
    const int C[3] = {13, 20, 5};
    const uint8_t luts[3][20] = {{4, 2, 2, 3, 3, 1, 2, 2, 2, 4, 4, 2, 4},
                                 {3, 3, 2, 2, 2, 2, 2, 2, 1, 3, 4, 4, 4, 2, 2, 2, 2, 2, 2, 4},
                                 {3, 1, 1, 2, 2}};
    const int64_t hw = H * W, npix = n_img * hw;
    Bench b;
    memset(&b.prm, 0, sizeof(b.prm));
    b.npix = npix;
    b.reps = reps;
    b.soak_s = soak;
    for (int s = 0; s < 3; ++s) {
        float *m, *a;
        const int64_t cnt = npix * C[s];
        if (cudaMalloc(&m, cnt * 4) != cudaSuccess || cudaMalloc(&a, cnt * 4) != cudaSuccess) { printf("alloc failed\n"); return 1; }
        fill_logits<<<148 * 8, 256>>>(m, a, cnt, 0x9e3779b9u * (s + 1), C[s], lowres ? hw / 4 : hw);
        b.prm.lr.hm[s] = (int)H / 2; b.prm.lr.wm[s] = (int)W / 2; b.prm.lr.ha[s] = (int)H / 4; b.prm.lr.wa[s] = (int)W / 4;
        b.prm.main[s] = m; b.prm.aux[s] = a; b.prm.C[s] = C[s];
        memcpy(b.prm.lut[s], luts[s], C[s]);
    }
    cudaMalloc(&b.prm.label, npix);
    cudaMalloc(&b.prm.conf, npix * 4);
    cudaMalloc(&b.prm.unc, npix * 4);
    cudaMalloc(&b.d_stats, sizeof(unsigned long long) * (8 + 8 + 8 * 2048 + 8));
    b.prm.S = 3; b.prm.K = 5; b.prm.policy = policy; b.prm.vote_t = vote_t; b.prm.ignore = 4; b.prm.ds_rate = 1;
    b.prm.n_img = n_img; b.prm.hw = hw;
    b.prm.class_hist = b.d_stats; b.prm.marginal = b.d_stats + 8; b.prm.conf_hist = hist ? b.d_stats + 16 : nullptr;
    if (cudaDeviceSynchronize() != cudaSuccess) { printf("init failed\n"); return 1; }
    const bool gk = policy == MSPL_POLICY_PROB || vote_t < 3;
    printf("# k1_sweep: %lld images %lldx%lld, 3 sources 13/20/5, policy=%d vote_t=%d gk=%d hist=%d, %.2f GB of logits\n", (long long)n_img,
           (long long)W, (long long)H, policy, vote_t, (int)gk, (int)hist, npix * 304.0 / 1e9);
    if (lowres) {
        // main at H/2 x W/2 and aux at H/4 x W/4 occupy the front of the full-size buffers allocated above
        b.prm.lr.H = (int)H; b.prm.lr.W = (int)W;
        if (!gk) {
            LOWRES(15, 2, 5, 4, false);
            LOWRES(15, 2, 5, 3, false);
            LOWRES(19, 2, 5, 3, false);
            LOWRES(11, 2, 5, 4, false);
        } else {
            LOWRES(15, 2, 5, 4, true);
            LOWRES(19, 2, 5, 3, true);
        }
        return 0;
    }
    if (!gk) {
        LABELS(15, 2, 5, 4);
        DIRECT(5, 256, 2, false);
        TMA(15, 2, 5, 4, false);
        TMA(15, 2, 5, 3, false);
        TMA(11, 2, 5, 5, false);
        TMA(19, 2, 5, 3, false);
        TMA(17, 2, 5, 3, false);
        TMA(23, 2, 5, 2, false);
        TMA(15, 2, 4, 5, false);
        TMA(15, 2, 7, 3, false);
        TMA(7, 2, 5, 8, false);
    } else {
        DIRECT(5, 256, 1, true);
        TMA(15, 2, 5, 4, true);
        TMA(15, 2, 5, 3, true);
        TMA(11, 2, 5, 5, true);
        TMA(19, 2, 5, 3, true);
        TMA(15, 2, 4, 5, true);
    }
    return 0;
}
