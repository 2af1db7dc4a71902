// Device-side building blocks shared by the forward and backward selective-scan kernels (sm_100a).
//
// Design (see DESIGN.md).  Persistent CTAs of 15 consumer warps + 1 producer warp.  Work is cut into SEGMENTS
// (batch b, B/C group g, a contiguous range of the group's rows).  For every (segment, chunk of <= 256 tokens)
// the producer stages one GROUP stage (the B and C chunk for all d_state rows + the per-row parameters
// A*log2e, D, delta_bias) and then streams the segment's rows through a ring of ROW stages (u, delta,
// [z, dout, out, h0]) -- all with 1-D TMA bulk copies (cp.async.bulk + mbarrier complete_tx), full/empty
// mbarrier pairs, no block-wide barrier in the steady state.  Consumer warps own rows: a row chunk is LPR lanes x
// 8 consecutive tokens, every lane scans its 8 tokens serially in registers, the lane aggregates are combined by
// a warp-shuffle scan of (a, b) pairs under (a, b) o (a', b') = (a a', a' b + b') (the algebra of
// selective_scan_common.h:91-96 in the reference), chunks are chained through shared-memory carries.
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "scan_args.h"

namespace mia {

constexpr float kLog2e = 1.4426950408889634f;
constexpr float kLn2 = 0.6931471805599453f;

// ------------------------------------------------------------------------------------------------
// PTX wrappers: mbarrier, TMA bulk copy, fast math.
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive(uint64_t *bar) {
    asm volatile("{\n\t.reg .b64 st;\n\tmbarrier.arrive.shared::cta.b64 st, [%0];\n\t}" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("{\n\t.reg .b64 st;\n\tmbarrier.arrive.expect_tx.shared::cta.b64 st, [%0], %1;\n\t}" ::"r"(smem_u32(bar)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "W_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra D_%=;\n\t"
        "bra W_%=;\n\t"
        "D_%=:\n\t}" ::"r"(smem_u32(bar)), "r"(parity)
        : "memory");
}
// 1-D TMA: global -> shared, completion signalled on an mbarrier (SASS: UBLKCP).
__device__ __forceinline__ void bulk_g2s(void *smem_dst, const void *gsrc, uint32_t bytes, uint64_t *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(smem_dst)),
                 "l"(gsrc), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}

__device__ __forceinline__ float ex2f(float x) { float y; asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float lg2f(float x) { float y; asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float rcpf(float x) { float y; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }

// softplus(x) = log1p(exp(x)) for x <= 20, x above (fwd_kernel_oflex.cuh:126), and optionally its derivative
// sigmoid(x) (bwd_kernel_oflex.cuh:252-257).  Evaluated as max(lg2(1 + 2^min(x log2e, 120)) ln2, x): for 20 < x the
// log1p term equals x to fp32 precision, the clamp keeps 2^. finite, the max restores x where the clamp bit.
// Absolute error <= 1 ulp of 1.0 (6e-8), which is what enters exp(dl A) and dl u B.
template <bool kWithSigmoid>
__device__ __forceinline__ float softplus_f(float x, float &sig) {
    const float e = ex2f(fminf(x * kLog2e, 120.f));
    const float s = 1.f + e;
    if (kWithSigmoid) sig = e * rcpf(s);
    return fmaxf(lg2f(s) * kLn2, x);
}

// ------------------------------------------------------------------------------------------------
// dtype traits + 8-token vector access with runtime alignment dispatch (the dispatch is warp-uniform
// for a row chunk because every lane sits a multiple of 16 (or 32) bytes from the row start).
template <typename T> struct Cvt;
template <> struct Cvt<float> {
    using raw = uint32_t;
    static __device__ __forceinline__ float to_f(raw v) { return __uint_as_float(v); }
    static __device__ __forceinline__ raw from_f(float v) { return __float_as_uint(v); }
};
template <> struct Cvt<__half> {
    using raw = uint16_t;
    static __device__ __forceinline__ float to_f(raw v) { return __half2float(__ushort_as_half(v)); }
    static __device__ __forceinline__ raw from_f(float v) { return __half_as_ushort(__float2half_rn(v)); }
};
template <> struct Cvt<__nv_bfloat16> {
    using raw = uint16_t;
    static __device__ __forceinline__ float to_f(raw v) { return __uint_as_float((uint32_t)v << 16); }
    static __device__ __forceinline__ raw from_f(float v) { return __bfloat16_as_ushort(__float2bfloat16_rn(v)); }
};

template <typename T> struct Pack8 { typename Cvt<T>::raw v[kTok]; };

// 8 consecutive T from a SHARED-memory address (32-bit shared-window address, element aligned) -> floats
template <typename T>
__device__ __forceinline__ void lds8(uint32_t saddr, float (&f)[kTok]) {
    constexpr int kBytes = kTok * (int)sizeof(T);
    union { Pack8<T> t; uint4 q[kBytes / 16]; uint2 d[kBytes / 8]; uint32_t w[kBytes / 4]; } buf;
    if ((saddr & 15) == 0) {
#pragma unroll
        for (int i = 0; i < kBytes / 16; ++i)
            asm volatile("ld.shared.v4.b32 {%0,%1,%2,%3}, [%4];" : "=r"(buf.q[i].x), "=r"(buf.q[i].y), "=r"(buf.q[i].z), "=r"(buf.q[i].w)
                         : "r"(saddr + 16 * i));
    } else if ((saddr & 7) == 0) {
#pragma unroll
        for (int i = 0; i < kBytes / 8; ++i)
            asm volatile("ld.shared.v2.b32 {%0,%1}, [%2];" : "=r"(buf.d[i].x), "=r"(buf.d[i].y) : "r"(saddr + 8 * i));
    } else if ((saddr & 3) == 0) {
#pragma unroll
        for (int i = 0; i < kBytes / 4; ++i) asm volatile("ld.shared.b32 %0, [%1];" : "=r"(buf.w[i]) : "r"(saddr + 4 * i));
    } else {
#pragma unroll
        for (int i = 0; i < kTok; ++i) {
            uint16_t h;
            asm volatile("ld.shared.u16 %0, [%1];" : "=h"(h) : "r"(saddr + 2 * i));
            buf.t.v[i] = (typename Cvt<T>::raw)h;
        }
    }
#pragma unroll
    for (int i = 0; i < kTok; ++i) f[i] = Cvt<T>::to_f(buf.t.v[i]);
}

// store up to 8 consecutive T to global memory (nvalid < 8 only in the lane that holds the sequence tail)
template <typename T>
__device__ __forceinline__ void st8(void *p, const float (&f)[kTok], int nvalid) {
    constexpr int kBytes = kTok * (int)sizeof(T);
    constexpr int kPer4 = 4 / (int)sizeof(T);       // elements per 32-bit word
    union { Pack8<T> t; uint4 q[kBytes / 16]; uint2 d[kBytes / 8]; uint32_t w[kBytes / 4]; } buf;
#pragma unroll
    for (int i = 0; i < kTok; ++i) buf.t.v[i] = Cvt<T>::from_f(f[i]);
    const uintptr_t a = (uintptr_t)p;
    if (nvalid >= kTok) {
        if ((a & 15) == 0) {
#pragma unroll
            for (int i = 0; i < kBytes / 16; ++i) reinterpret_cast<uint4 *>(p)[i] = buf.q[i];
            return;
        } else if ((a & 7) == 0) {
#pragma unroll
            for (int i = 0; i < kBytes / 8; ++i) reinterpret_cast<uint2 *>(p)[i] = buf.d[i];
            return;
        }
    }
    if ((a & 3) == 0) {   // word stores for the full words, then at most one trailing element
#pragma unroll
        for (int i = 0; i < kBytes / 4; ++i)
            if ((i + 1) * kPer4 <= nvalid) reinterpret_cast<uint32_t *>(p)[i] = buf.w[i];
        if (kPer4 == 2 && (nvalid & 1)) reinterpret_cast<typename Cvt<T>::raw *>(p)[nvalid - 1] = buf.t.v[(nvalid - 1) & 7];
        return;
    }
#pragma unroll
    for (int i = 0; i < kTok; ++i)
        if (i < nvalid) reinterpret_cast<typename Cvt<T>::raw *>(p)[i] = buf.t.v[i];
}

// ------------------------------------------------------------------------------------------------
// Packed f32x2 arithmetic (sm_100: FFMA2 / FMUL2 / FADD2 -- two fp32 lanes per issued instruction) and the
// 8-token <-> 4 x float2 conversions the fast paths are written in.
__device__ __forceinline__ float2 fma2(float2 a, float2 b, float2 c) { return __ffma2_rn(a, b, c); }
__device__ __forceinline__ float2 mul2(float2 a, float2 b) { return __fmul2_rn(a, b); }
__device__ __forceinline__ float2 add2(float2 a, float2 b) { return __fadd2_rn(a, b); }
__device__ __forceinline__ float2 splat2(float v) { return make_float2(v, v); }

template <int kWords>
__device__ __forceinline__ void lds_words(uint32_t saddr, uint32_t (&w)[kWords]) {
    if ((saddr & 15) == 0) {
#pragma unroll
        for (int i = 0; i < kWords / 4; ++i)
            asm volatile("ld.shared.v4.b32 {%0,%1,%2,%3}, [%4];" : "=r"(w[4 * i]), "=r"(w[4 * i + 1]), "=r"(w[4 * i + 2]), "=r"(w[4 * i + 3])
                         : "r"(saddr + 16 * i));
    } else if ((saddr & 7) == 0) {
#pragma unroll
        for (int i = 0; i < kWords / 2; ++i)
            asm volatile("ld.shared.v2.b32 {%0,%1}, [%2];" : "=r"(w[2 * i]), "=r"(w[2 * i + 1]) : "r"(saddr + 8 * i));
    } else if ((saddr & 3) == 0) {
#pragma unroll
        for (int i = 0; i < kWords; ++i) asm volatile("ld.shared.b32 %0, [%1];" : "=r"(w[i]) : "r"(saddr + 4 * i));
    } else {   // 2-byte aligned (16-bit types with odd sequence length)
#pragma unroll
        for (int i = 0; i < kWords; ++i) {
            uint16_t lo, hi;
            asm volatile("ld.shared.u16 %0, [%1];" : "=h"(lo) : "r"(saddr + 4 * i));
            asm volatile("ld.shared.u16 %0, [%1];" : "=h"(hi) : "r"(saddr + 4 * i + 2));
            w[i] = (uint32_t)lo | ((uint32_t)hi << 16);
        }
    }
}

template <typename T> struct Vec;   // 8 tokens as 4 float2
template <> struct Vec<__nv_bfloat16> {
    static constexpr int kWords = 4;
    static __device__ __forceinline__ float2 up(uint32_t w) { return make_float2(__uint_as_float(w << 16), __uint_as_float(w & 0xffff0000u)); }
    static __device__ __forceinline__ void unpack(const uint32_t (&w)[4], float2 (&f)[4]) {
#pragma unroll
        for (int k = 0; k < 4; ++k) f[k] = up(w[k]);
    }
    static __device__ __forceinline__ void pack(const float2 (&f)[4], uint32_t (&w)[4]) {
#pragma unroll
        for (int k = 0; k < 4; ++k) { __nv_bfloat162 h = __floats2bfloat162_rn(f[k].x, f[k].y); w[k] = *reinterpret_cast<uint32_t *>(&h); }
    }
};
template <> struct Vec<__half> {
    static constexpr int kWords = 4;
    static __device__ __forceinline__ void unpack(const uint32_t (&w)[4], float2 (&f)[4]) {
#pragma unroll
        for (int k = 0; k < 4; ++k) { __half2 h = *reinterpret_cast<const __half2 *>(&w[k]); f[k] = __half22float2(h); }
    }
    static __device__ __forceinline__ void pack(const float2 (&f)[4], uint32_t (&w)[4]) {
#pragma unroll
        for (int k = 0; k < 4; ++k) { __half2 h = __floats2half2_rn(f[k].x, f[k].y); w[k] = *reinterpret_cast<uint32_t *>(&h); }
    }
};
template <> struct Vec<float> {
    static constexpr int kWords = 8;
    static __device__ __forceinline__ void unpack(const uint32_t (&w)[8], float2 (&f)[4]) {
#pragma unroll
        for (int k = 0; k < 4; ++k) f[k] = make_float2(__uint_as_float(w[2 * k]), __uint_as_float(w[2 * k + 1]));
    }
    static __device__ __forceinline__ void pack(const float2 (&f)[4], uint32_t (&w)[8]) {
#pragma unroll
        for (int k = 0; k < 4; ++k) { w[2 * k] = __float_as_uint(f[k].x); w[2 * k + 1] = __float_as_uint(f[k].y); }
    }
};

template <typename T>
__device__ __forceinline__ void lds8v(uint32_t saddr, float2 (&f)[4]) {
    uint32_t w[Vec<T>::kWords];
    lds_words<Vec<T>::kWords>(saddr, w);
    Vec<T>::unpack(w, f);
}

// store 8 tokens (nvalid of them) to global memory with the widest stores the address allows
template <typename T>
__device__ __forceinline__ void st8v(void *p, const float2 (&f)[4], int nvalid) {
    constexpr int kWords = Vec<T>::kWords;
    constexpr int kPer = 8 / kWords;     // tokens per 32-bit word
    uint32_t w[kWords];
    Vec<T>::pack(f, w);
    const uintptr_t a = (uintptr_t)p;
    if (nvalid >= kTok) {
        if ((a & 15) == 0) {
#pragma unroll
            for (int i = 0; i < kWords / 4; ++i) reinterpret_cast<uint4 *>(p)[i] = make_uint4(w[4 * i], w[4 * i + 1], w[4 * i + 2], w[4 * i + 3]);
            return;
        } else if ((a & 7) == 0) {
#pragma unroll
            for (int i = 0; i < kWords / 2; ++i) reinterpret_cast<uint2 *>(p)[i] = make_uint2(w[2 * i], w[2 * i + 1]);
            return;
        }
    }
    if ((a & 3) == 0) {
#pragma unroll
        for (int i = 0; i < kWords; ++i)
            if ((i + 1) * kPer <= nvalid) reinterpret_cast<uint32_t *>(p)[i] = w[i];
        if (kPer == 2 && (nvalid & 1) && nvalid < kTok) {
#pragma unroll
            for (int i = 0; i < kWords; ++i)
                if (2 * i + 1 == nvalid) reinterpret_cast<uint16_t *>(p)[2 * i] = (uint16_t)(w[i] & 0xffffu);
        }
        return;
    }
    if (kPer == 2) {
#pragma unroll
        for (int i = 0; i < kTok; ++i)
            if (i < nvalid) reinterpret_cast<uint16_t *>(p)[i] = (uint16_t)((w[i >> 1] >> ((i & 1) * 16)) & 0xffffu);
    }
}

// ------------------------------------------------------------------------------------------------
// Producer side: copy `nbytes` from global `src` into the shared slot so that source byte k lands at
// slot + (src & 15) + k.  The 16-byte-aligned interior goes through one TMA bulk copy; the (< 16 B) head and
// tail are copied element-wise by the calling lane.  Returns the bytes the bulk copy will complete on `bar`.
__device__ __forceinline__ uint32_t stage_span(char *slot, const char *src, uint32_t nbytes, uint64_t *bar, int esize) {
    const uint32_t mis = (uint32_t)((uintptr_t)src & 15u);
    char *dst = slot + mis;
    uint32_t head = mis ? (16u - mis) : 0u;
    if (head > nbytes) head = nbytes;
    const uint32_t body = (nbytes - head) & ~15u;
    const uint32_t tail = nbytes - head - body;
    if (body) bulk_g2s(dst + head, src + head, body, bar);
    if (esize == 2) {
        for (uint32_t k = 0; k < head; k += 2) *reinterpret_cast<uint16_t *>(dst + k) = *reinterpret_cast<const uint16_t *>(src + k);
        for (uint32_t k = head + body; k < head + body + tail; k += 2)
            *reinterpret_cast<uint16_t *>(dst + k) = *reinterpret_cast<const uint16_t *>(src + k);
    } else {
        for (uint32_t k = 0; k < head; k += 4) *reinterpret_cast<uint32_t *>(dst + k) = *reinterpret_cast<const uint32_t *>(src + k);
        for (uint32_t k = head + body; k < head + body + tail; k += 4)
            *reinterpret_cast<uint32_t *>(dst + k) = *reinterpret_cast<const uint32_t *>(src + k);
    }
    return body;
}

// Stage `nrows` row chunks of `len` elements each (element size es, global row stride row_stride elements).
// flat: the rows are back to back in global memory (row_stride == len) -> a single span.
__device__ __forceinline__ uint32_t stage_rows(char *region, const char *g0, long long row_stride, int nrows, int len, int es,
                                               int pitch, bool flat, uint64_t *bar, int lane) {
    uint32_t tx = 0;
    if (flat) {
        if (lane == 0) tx = stage_span(region, g0, (uint32_t)nrows * len * es, bar, es);
    } else {
        for (int r = lane; r < nrows; r += 32)
            tx += stage_span(region + (size_t)r * pitch, g0 + (size_t)r * row_stride * es, (uint32_t)len * es, bar, es);
    }
    return tx;
}

// Consumer side view of a region staged by stage_rows: row r starts at base + r * pitch + ((g0lo + r * gstep) & 15).
// (flat: pitch = len * es, gstep = 0, so the misalignment is that of the tile start.)
struct RowView {
    uint32_t base, pitch, g0lo, gstep;
    __device__ __forceinline__ uint32_t row(int r) const { return base + r * pitch + ((g0lo + r * gstep) & 15u); }
};
__device__ __forceinline__ RowView make_view(const char *region, const char *g0, long long row_stride, int len, int es, int pitch,
                                             bool flat) {
    RowView v;
    v.base = smem_u32(region);
    v.g0lo = (uint32_t)(uintptr_t)g0;
    if (flat) { v.pitch = (uint32_t)(len * es); v.gstep = 0; }
    else { v.pitch = (uint32_t)pitch; v.gstep = (uint32_t)(row_stride * es); }
    return v;
}

struct SegCoord { int b, g, row_lo, nrows; };
__device__ __forceinline__ SegCoord decode_seg(const ScanArgs &a, int seg) {
    SegCoord c;
    const int s = seg % a.split;
    const int bg = seg / a.split;
    c.g = bg % a.G;
    c.b = bg / a.G;
    const int in_group = s * a.RS;
    c.row_lo = c.g * a.rows_per_group + in_group;
    c.nrows = min(a.RS, a.rows_per_group - in_group);
    return c;
}

// ------------------------------------------------------------------------------------------------
// Warp-shuffle scans of (a, b) pairs over segments of `lpr` lanes (lpr is a power of two, j = lane % lpr).
// kLPR == 32: the row is the whole warp, everything unrolls without width bookkeeping; kLPR == 0: runtime lpr.
// Forward: on return (pa, pb) is the inclusive aggregate of lanes [0..j]; (ea, eb) the exclusive one.
template <int kLPR>
__device__ __forceinline__ void seg_scan_fwd(float &pa, float &pb, float &ea, float &eb, int j, int lpr) {
    if (kLPR == 32) {
#pragma unroll
        for (int off = 1; off < 32; off <<= 1) {
            float qa = __shfl_up_sync(0xffffffffu, pa, off);
            float qb = __shfl_up_sync(0xffffffffu, pb, off);
            const bool ok = j >= off;
            qa = ok ? qa : 1.f;
            qb = ok ? qb : 0.f;
            pb = fmaf(pa, qb, pb);   // earlier piece (qa,qb) then ours (pa,pb): (qa pa, pa qb + pb)
            pa = pa * qa;
        }
        ea = __shfl_up_sync(0xffffffffu, pa, 1);
        eb = __shfl_up_sync(0xffffffffu, pb, 1);
    } else {
        for (int off = 1; off < lpr; off <<= 1) {
            float qa = __shfl_up_sync(0xffffffffu, pa, off, lpr);
            float qb = __shfl_up_sync(0xffffffffu, pb, off, lpr);
            const bool ok = j >= off;
            qa = ok ? qa : 1.f;
            qb = ok ? qb : 0.f;
            pb = fmaf(pa, qb, pb);
            pa = pa * qa;
        }
        ea = __shfl_up_sync(0xffffffffu, pa, 1, lpr);
        eb = __shfl_up_sync(0xffffffffu, pb, 1, lpr);
    }
    if (j == 0) { ea = 1.f; eb = 0.f; }
}
// Reverse (suffix) scan: G_t = rb_t + ra_t * G_{t+1}.  On return (pa, pb) aggregates lanes [j..lpr-1],
// (ea, eb) lanes [j+1..lpr-1].
template <int kLPR>
__device__ __forceinline__ void seg_scan_rev(float &pa, float &pb, float &ea, float &eb, int j, int lpr) {
    if (kLPR == 32) {
#pragma unroll
        for (int off = 1; off < 32; off <<= 1) {
            float qa = __shfl_down_sync(0xffffffffu, pa, off);
            float qb = __shfl_down_sync(0xffffffffu, pb, off);
            const bool ok = j + off < 32;
            qa = ok ? qa : 1.f;
            qb = ok ? qb : 0.f;
            pb = fmaf(pa, qb, pb);
            pa = pa * qa;
        }
        ea = __shfl_down_sync(0xffffffffu, pa, 1);
        eb = __shfl_down_sync(0xffffffffu, pb, 1);
    } else {
        for (int off = 1; off < lpr; off <<= 1) {
            float qa = __shfl_down_sync(0xffffffffu, pa, off, lpr);
            float qb = __shfl_down_sync(0xffffffffu, pb, off, lpr);
            const bool ok = j + off < lpr;
            qa = ok ? qa : 1.f;
            qb = ok ? qb : 0.f;
            pb = fmaf(pa, qb, pb);
            pa = pa * qa;
        }
        ea = __shfl_down_sync(0xffffffffu, pa, 1, lpr);
        eb = __shfl_down_sync(0xffffffffu, pb, 1, lpr);
    }
    if (j == lpr - 1) { ea = 1.f; eb = 0.f; }
}

// sum over the lanes of a row piece; result valid in every lane of the piece
template <int kLPR>
__device__ __forceinline__ float seg_sum(float v, int lpr) {
    if (kLPR == 32) {
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
    } else {
        for (int off = lpr >> 1; off > 0; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off, 32);
    }
    return v;
}
// three full-warp sums for the price of six shuffles: on return lane 0 holds sum(a), lane 16 sum(b), lane 8 sum(c)
__device__ __forceinline__ float warp_sum3(float a, float b, float c, int lane) {
    const bool hi = lane & 16;
    float p = (hi ? b : a) + __shfl_xor_sync(0xffffffffu, hi ? a : b, 16);   // lo half: a pairs, hi half: b pairs
    float q = c + __shfl_xor_sync(0xffffffffu, c, 16);                        // both halves: c pairs
    const bool b3 = lane & 8;
    float r = (b3 ? q : p) + __shfl_xor_sync(0xffffffffu, b3 ? p : q, 8);    // bit3 = 0: a|b quads, bit3 = 1: c quads
    r += __shfl_xor_sync(0xffffffffu, r, 4);
    r += __shfl_xor_sync(0xffffffffu, r, 2);
    r += __shfl_xor_sync(0xffffffffu, r, 1);
    return r;
}

// zero the dynamic shared memory once per CTA so that padding / not-yet-written bytes read as finite values
__device__ __forceinline__ void zero_smem(char *smem, int bytes) {
    uint4 *p = reinterpret_cast<uint4 *>(smem);
    for (int i = threadIdx.x; i < bytes / 16; i += blockDim.x) p[i] = make_uint4(0, 0, 0, 0);
    fence_proxy_async();
}

}  // namespace mia
