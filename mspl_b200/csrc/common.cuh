// Shared device/host helpers for the mspl_b200 kernels (sm_100a).
#pragma once
#include <cuda_runtime.h>
#include <cuda_fp16.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <math.h>
#include <initializer_list>

#include "../../include/mspl_b200.h"

namespace mspl {

constexpr int kNumSMs = 148;            // B200: 2 dies x 74 SMs
constexpr float kLog2e = 1.4426950408889634f;
constexpr float kNearTieMargin = 1e-6f; // BASELINE.json north_star: top-2 probability margin of a "marginal" pixel

#define MSPL_DEVINL __device__ __forceinline__

// ---- streaming vector access: P consecutive fp32 pixels of one class plane -------------------------
// Inputs are read exactly once, so they bypass L1 allocation (ld.global.nc.L1::no_allocate).
template <int P> struct PixVec;
template <> struct PixVec<1> {
    static MSPL_DEVINL void load(const float* p, float (&v)[1]) {
        asm volatile("ld.global.nc.L1::no_allocate.f32 %0, [%1];" : "=f"(v[0]) : "l"(p));
    }
    static MSPL_DEVINL void store(float* p, const float (&v)[1]) { __stcs(p, v[0]); }
};
template <> struct PixVec<2> {
    static MSPL_DEVINL void load(const float* p, float (&v)[2]) {
        asm volatile("ld.global.nc.L1::no_allocate.v2.f32 {%0,%1}, [%2];" : "=f"(v[0]), "=f"(v[1]) : "l"(p));
    }
    static MSPL_DEVINL void store(float* p, const float (&v)[2]) {
        __stcs(reinterpret_cast<float2*>(p), make_float2(v[0], v[1]));
    }
};
template <> struct PixVec<4> {
    static MSPL_DEVINL void load(const float* p, float (&v)[4]) {
        asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
                     : "=f"(v[0]), "=f"(v[1]), "=f"(v[2]), "=f"(v[3]) : "l"(p));
    }
    static MSPL_DEVINL void store(float* p, const float (&v)[4]) {
        __stcs(reinterpret_cast<float4*>(p), make_float4(v[0], v[1], v[2], v[3]));
    }
};

// ---- the same for fp16 / bf16 planes (autocast logits): loads upcast to fp32, which is exact; stores round to nearest even
template <typename LT> MSPL_DEVINL float half_to_float(uint32_t bits);
template <> MSPL_DEVINL float half_to_float<__half>(uint32_t bits) { return __half2float(__ushort_as_half((unsigned short)bits)); }
template <> MSPL_DEVINL float half_to_float<__nv_bfloat16>(uint32_t bits) { return __uint_as_float(bits << 16); }
template <typename LT> MSPL_DEVINL uint32_t float_to_half(float f);
template <> MSPL_DEVINL uint32_t float_to_half<__half>(float f) { return __half_as_ushort(__float2half_rn(f)); }
template <> MSPL_DEVINL uint32_t float_to_half<__nv_bfloat16>(float f) { return __bfloat16_as_ushort(__float2bfloat16_rn(f)); }

// P consecutive 2-byte pixels of one class plane, P in {1, 2, 4}: one 2-, 4- or 8-byte access.
template <typename LT, int P> struct HalfVec {
    static MSPL_DEVINL void load(const LT* p, float (&v)[P]) {
        uint32_t w[(P + 1) / 2];
        if (P == 1) {
            unsigned short b;
            asm volatile("ld.global.nc.L1::no_allocate.b16 %0, [%1];" : "=h"(b) : "l"(p));
            w[0] = b;
        } else if (P == 2) {
            asm volatile("ld.global.nc.L1::no_allocate.b32 %0, [%1];" : "=r"(w[0]) : "l"(p));
        } else {
            asm volatile("ld.global.nc.L1::no_allocate.v2.b32 {%0,%1}, [%2];" : "=r"(w[0]), "=r"(w[P > 2 ? 1 : 0]) : "l"(p));
        }
#pragma unroll
        for (int i = 0; i < P; ++i) v[i] = half_to_float<LT>((w[i / 2] >> (16 * (i & 1))) & 0xffffu);
    }
    static MSPL_DEVINL void store(LT* p, const float (&v)[P]) {
        uint32_t w[(P + 1) / 2];
#pragma unroll
        for (int i = 0; i < (P + 1) / 2; ++i)
            w[i] = float_to_half<LT>(v[2 * i]) | (2 * i + 1 < P ? float_to_half<LT>(v[(2 * i + 1) % P]) << 16 : 0u);
        if (P == 1) {
            asm volatile("st.global.cs.b16 [%0], %1;" ::"l"(p), "h"((unsigned short)w[0]) : "memory");
        } else if (P == 2) {
            asm volatile("st.global.cs.b32 [%0], %1;" ::"l"(p), "r"(w[0]) : "memory");
        } else {
            asm volatile("st.global.cs.v2.b32 [%0], {%1,%2};" ::"l"(p), "r"(w[0]), "r"(w[P > 2 ? 1 : 0]) : "memory");
        }
    }
};

// Logit planes of element type LT: fp32 through PixVec, fp16 / bf16 through HalfVec.
template <typename LT, int P> struct LogitVec : HalfVec<LT, P> {};
template <int P> struct LogitVec<float, P> : PixVec<P> {};

template <int P> MSPL_DEVINL void store_labels(uint8_t* p, const int (&l)[P]);
template <> MSPL_DEVINL void store_labels<1>(uint8_t* p, const int (&l)[1]) { p[0] = (uint8_t)l[0]; }
template <> MSPL_DEVINL void store_labels<2>(uint8_t* p, const int (&l)[2]) {
    *reinterpret_cast<uchar2*>(p) = make_uchar2((uint8_t)l[0], (uint8_t)l[1]);
}
template <> MSPL_DEVINL void store_labels<4>(uint8_t* p, const int (&l)[4]) {
    *reinterpret_cast<uchar4*>(p) = make_uchar4((uint8_t)l[0], (uint8_t)l[1], (uint8_t)l[2], (uint8_t)l[3]);
}

// exp(x - M) with one FFMA + one MUFU.EX2: callers pass x and Ml = M*log2e.
MSPL_DEVINL float exp_shifted(float x, float Ml) { return exp2f(fmaf(x, kLog2e, -Ml)); }

// Order-preserving map fp32 -> u32 (larger float <=> larger key) and back; used by the radix select.
MSPL_DEVINL uint32_t float_to_key(float f) {
    const uint32_t b = __float_as_uint(f);
    return b ^ ((uint32_t)((int32_t)b >> 31) | 0x80000000u);      // negative: flip all bits; else set the sign bit
}
MSPL_DEVINL float key_to_float(uint32_t k) {
    uint32_t b = (k & 0x80000000u) ? (k & 0x7fffffffu) : ~k;
    return __uint_as_float(b);
}
// digit of `key` examined by radix pass 0/1/2 (11 + 11 + 10 bits) and the prefix above it
MSPL_DEVINL uint32_t radix_digit(uint32_t key, int pass) {
    return pass == 0 ? (key >> 21) : pass == 1 ? ((key >> 10) & 0x7ffu) : (key & 0x3ffu);
}
MSPL_DEVINL uint32_t radix_prefix(uint32_t key, int pass) {
    return pass == 0 ? 0u : pass == 1 ? (key >> 21) : (key >> 10);
}

// Bin of the LINEAR confidence histogram (MSPL_RADIX_BINS equal steps over [0,1], clamped): monotone non-decreasing in f
// for every float (x2048 is exact), so "bin above / below the class's selected bin" brackets the order statistic.
// bin(f) >= b  <=>  f >= b/2048 for 1 <= b <= 2047 (both sides exact in fp32).  NaN lands in bin 0.
MSPL_DEVINL uint32_t conf_bin(float f) {
    return (uint32_t)max(0, min(MSPL_RADIX_BINS - 1, __float2int_rd(f * (float)MSPL_RADIX_BINS)));
}

MSPL_DEVINL double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

inline bool aligned_to(const void* p, size_t a) { return (reinterpret_cast<uintptr_t>(p) % a) == 0; }

inline int launch_status() { return cudaPeekAtLastError() == cudaSuccess ? MSPL_OK : MSPL_ERR_CUDA; }

// Largest pixel vector width usable for planes of `hw` floats starting at the given bases.
inline int pick_vec(int64_t hw, std::initializer_list<const void*> ptrs) {
    int p = (hw % 4 == 0) ? 4 : (hw % 2 == 0) ? 2 : 1;
    for (const void* q : ptrs) {
        if (!q) continue;
        while (p > 1 && !aligned_to(q, 4 * p)) p >>= 1;
    }
    return p;
}

}  // namespace mspl
