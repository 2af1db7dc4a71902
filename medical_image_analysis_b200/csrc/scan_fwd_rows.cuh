// Forward selective scan, ROW-SERIAL path (d_state == 1): one LANE per row, tokens walked serially.
//
// Why: with one state per row the warp-scan formulation spends most of its issue slots on the scan itself, on
// per-row bookkeeping and on lanes idling past the end of a 196-token row (profiles/README.md).  Here a warp owns 32
// consecutive rows; every lane runs the recurrence h = a h + b of its own row in a register -- no shuffles, no lane
// idles, ~15 instructions per token -- and the 32 rows advance in lock step, so B[t], C[t] are shared-memory
// broadcasts.  Each warp is its own pipeline (no block-wide state at all):
//   * lane 0 TMA-loads the next [32 rows x chunk] tiles of u and delta (one flat bulk copy each when the chunk is the
//     whole row, else one per row) and the B / C chunk into the other half of a warp-private double buffer;
//   * y overwrites u in shared memory and leaves with ONE bulk store (cp.async.bulk.global.shared::cta) -> coalesced
//     128-byte writes although every lane produces a different row;
//   * (prod a, h) is checkpointed into x at the same 256-token boundaries as the warp-scan kernels, so either
//     backward kernel can consume it.
// Preconditions (checked on the host, otherwise the warp-scan kernels run): d_state == 1, delta per row, no z,
// rows contiguous (stride == L), rows_per_group % 32 == 0, chunk % 4 == 0, 16-byte aligned tiles.
#pragma once
#include <type_traits>

#include "scan_common.cuh"

namespace mia {

__device__ __forceinline__ void bulk_s2g(void *gdst, const void *ssrc, uint32_t bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gdst), "r"(smem_u32(ssrc)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int kN> __device__ __forceinline__ void bulk_wait_read() { asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(kN) : "memory"); }

// 4 consecutive tokens of T in shared memory <-> 2 float2 (8-byte aligned for 2-byte T, 16 for float).  Plain typed
// accesses (no asm): the compiler must see the dependences so that it can hoist the loads of later tokens above the
// in-place store of earlier ones and software-pipeline the token loop.
template <typename T> struct Quad;
template <> struct Quad<__nv_bfloat16> {
    static __device__ __forceinline__ void ld(const char *p, float2 (&f)[2]) {
        const uint2 w = *reinterpret_cast<const uint2 *>(p);
        f[0] = make_float2(__uint_as_float(w.x << 16), __uint_as_float(w.x & 0xffff0000u));
        f[1] = make_float2(__uint_as_float(w.y << 16), __uint_as_float(w.y & 0xffff0000u));
    }
    static __device__ __forceinline__ void st(char *p, const float2 (&f)[2]) {
        __nv_bfloat162 h0 = __floats2bfloat162_rn(f[0].x, f[0].y), h1 = __floats2bfloat162_rn(f[1].x, f[1].y);
        *reinterpret_cast<uint2 *>(p) = make_uint2(*reinterpret_cast<uint32_t *>(&h0), *reinterpret_cast<uint32_t *>(&h1));
    }
};
template <> struct Quad<__half> {
    static __device__ __forceinline__ void ld(const char *p, float2 (&f)[2]) {
        uint2 w = *reinterpret_cast<const uint2 *>(p);
        f[0] = __half22float2(*reinterpret_cast<__half2 *>(&w.x));
        f[1] = __half22float2(*reinterpret_cast<__half2 *>(&w.y));
    }
    static __device__ __forceinline__ void st(char *p, const float2 (&f)[2]) {
        __half2 h0 = __floats2half2_rn(f[0].x, f[0].y), h1 = __floats2half2_rn(f[1].x, f[1].y);
        *reinterpret_cast<uint2 *>(p) = make_uint2(*reinterpret_cast<uint32_t *>(&h0), *reinterpret_cast<uint32_t *>(&h1));
    }
};
template <> struct Quad<float> {
    static __device__ __forceinline__ void ld(const char *p, float2 (&f)[2]) {
        const float4 w = *reinterpret_cast<const float4 *>(p);
        f[0] = make_float2(w.x, w.y);
        f[1] = make_float2(w.z, w.w);
    }
    static __device__ __forceinline__ void st(char *p, const float2 (&f)[2]) {
        *reinterpret_cast<float4 *>(p) = make_float4(f[0].x, f[0].y, f[1].x, f[1].y);
    }
};

// 8 consecutive tokens of a 2-byte T (16 bytes, 16-byte aligned) <-> 4 float2.  Used on the swizzled TMA tiles of the
// column-walk kernels: there the 32 lanes of a warp read the same column of 32 different tile rows, the swizzle permutes the
// 16-byte chunks of 8 consecutive rows over one 128-byte bank line, and a 16-byte access per lane is conflict-free (each
// quarter-warp covers the line exactly once), while 8-byte accesses hit every 8-byte bank pair twice per half-warp (ncu of the
// quad version: a third of the shared-memory wavefronts of both kernels were bank conflicts, profiles/r2z_ncu_summary.json).
template <typename T> struct Oct;
template <> struct Oct<__nv_bfloat16> {
    static __device__ __forceinline__ void ld(const char *p, float2 (&f)[4]) {
        const uint4 w = *reinterpret_cast<const uint4 *>(p);
        f[0] = make_float2(__uint_as_float(w.x << 16), __uint_as_float(w.x & 0xffff0000u));
        f[1] = make_float2(__uint_as_float(w.y << 16), __uint_as_float(w.y & 0xffff0000u));
        f[2] = make_float2(__uint_as_float(w.z << 16), __uint_as_float(w.z & 0xffff0000u));
        f[3] = make_float2(__uint_as_float(w.w << 16), __uint_as_float(w.w & 0xffff0000u));
    }
    static __device__ __forceinline__ void st(char *p, const float2 (&f)[4]) {
        __nv_bfloat162 h0 = __floats2bfloat162_rn(f[0].x, f[0].y), h1 = __floats2bfloat162_rn(f[1].x, f[1].y),
                       h2 = __floats2bfloat162_rn(f[2].x, f[2].y), h3 = __floats2bfloat162_rn(f[3].x, f[3].y);
        *reinterpret_cast<uint4 *>(p) = make_uint4(*reinterpret_cast<uint32_t *>(&h0), *reinterpret_cast<uint32_t *>(&h1),
                                                   *reinterpret_cast<uint32_t *>(&h2), *reinterpret_cast<uint32_t *>(&h3));
    }
};
template <> struct Oct<__half> {
    static __device__ __forceinline__ void ld(const char *p, float2 (&f)[4]) {
        uint4 w = *reinterpret_cast<const uint4 *>(p);
        f[0] = __half22float2(*reinterpret_cast<__half2 *>(&w.x));
        f[1] = __half22float2(*reinterpret_cast<__half2 *>(&w.y));
        f[2] = __half22float2(*reinterpret_cast<__half2 *>(&w.z));
        f[3] = __half22float2(*reinterpret_cast<__half2 *>(&w.w));
    }
    static __device__ __forceinline__ void st(char *p, const float2 (&f)[4]) {
        __half2 h0 = __floats2half2_rn(f[0].x, f[0].y), h1 = __floats2half2_rn(f[1].x, f[1].y), h2 = __floats2half2_rn(f[2].x, f[2].y),
                h3 = __floats2half2_rn(f[3].x, f[3].y);
        *reinterpret_cast<uint4 *>(p) = make_uint4(*reinterpret_cast<uint32_t *>(&h0), *reinterpret_cast<uint32_t *>(&h1),
                                                   *reinterpret_cast<uint32_t *>(&h2), *reinterpret_cast<uint32_t *>(&h3));
    }
};
template <> struct Oct<float> {                  // (two 16-byte accesses; fp32 tiles are conflict-free per quad already)
    static __device__ __forceinline__ void ld(const char *, float2 (&)[4]) {}
    static __device__ __forceinline__ void st(char *, const float2 (&)[4]) {}
};

template <typename T, bool kSoftplus, bool kOutF32>
__global__ void __launch_bounds__(32) ss_fwd_rows_kernel(const __grid_constant__ RowsArgs a) {
    extern __shared__ __align__(128) char smem[];
    constexpr int es = (int)sizeof(T);
    const int lane = threadIdx.x;
    // layout: [u tile][delta tile][B ln2 as fp32][C as fp32][mbarrier]
    char *tu = smem, *td = smem + a.tile_bytes;
    float *Bf = reinterpret_cast<float *>(smem + a.off_bc32), *Cf = Bf + a.Lc;
    uint64_t *full = reinterpret_cast<uint64_t *>(smem + a.stage_bytes);
    if (lane == 0) { mbar_init(full, 1); fence_mbar_init(); }
    __syncwarp();

    const int L = a.L, Lc = a.Lc, nch = a.n_lchunks;
    const int batches_per_group = a.rows_per_group / 32;
    const float *Ap = reinterpret_cast<const float *>(a.A);
    const float *Dp = reinterpret_cast<const float *>(a.D);
    const float *biasp = reinterpret_cast<const float *>(a.delta_bias);
    const float2 kL2E = splat2(kLog2e), kOne = splat2(1.f);
    const uint32_t rowpitch = (uint32_t)((nch == 1 ? L : Lc) * es);
    char *pu = tu + lane * rowpitch;
    const char *pd = td + lane * rowpitch;
    uint32_t phase = 0;

    for (int item = blockIdx.x; item < a.n_items; item += gridDim.x) {
        const int bt = item % batches_per_group;
        const int bg = item / batches_per_group;
        const int g = bg % a.G, b = bg / a.G;
        const int row0 = g * a.rows_per_group + bt * 32;
        const int d = row0 + lane;
        const float Araw = __ldg(Ap + d);
        const float Dv = Dp ? __ldg(Dp + d) : 0.f;
        const float2 bl2 = splat2((biasp ? __ldg(biasp + d) : 0.f) * kLog2e), A2 = splat2(Araw), D2 = splat2(Dv);
        float h = 0.f;                           // recurrence state of this lane's row, carried across the chunks of the row
        float2 msum = make_float2(0.f, 0.f);     // sum of softplus * log2e so far (prod a = 2^(A * sum))
        float2 *xrow = reinterpret_cast<float2 *>(a.x) + ((size_t)b * a.dim + d) * a.xchunks;
        int xc = 0, to_ck = min(a.xchunk_tokens, L);   // next checkpoint slot, tokens until it is due
        for (int c = 0; c < nch; ++c) {
            const int l0 = c * Lc, len = min(Lc, L - l0);
            // ---- stage: u / delta tiles by TMA (one flat 32-row span when the chunk is the whole row, else one piece per
            //      row), B / C straight from global memory (coalesced, converted to fp32 once for the 32 rows)
            const char *gu = (const char *)a.u + (((size_t)b * a.dim + row0) * L + l0) * es;
            const char *gd = (const char *)a.delta + (((size_t)b * a.dim + row0) * L + l0) * es;
            if (nch == 1) {
                if (lane == 0) {
                    bulk_g2s(tu, gu, (uint32_t)(32 * L * es), full);
                    bulk_g2s(td, gd, (uint32_t)(32 * L * es), full);
                    mbar_arrive_expect_tx(full, 2u * 32u * L * es);
                }
            } else {
                bulk_g2s(tu + (size_t)lane * Lc * es, gu + (size_t)lane * L * es, (uint32_t)(len * es), full);
                bulk_g2s(td + (size_t)lane * Lc * es, gd + (size_t)lane * L * es, (uint32_t)(len * es), full);
                __syncwarp();
                if (lane == 0) mbar_arrive_expect_tx(full, 64u * len * es);
            }
            {
                const typename Cvt<T>::raw *gB = reinterpret_cast<const typename Cvt<T>::raw *>(a.B) + (size_t)b * a.B_bs + (size_t)g * a.B_gs + l0;
                const typename Cvt<T>::raw *gC = reinterpret_cast<const typename Cvt<T>::raw *>(a.C) + (size_t)b * a.C_bs + (size_t)g * a.C_gs + l0;
                for (int i = lane; i < len; i += 32) {
                    Bf[i] = Cvt<T>::to_f(__ldg(gB + i)) * kLn2;
                    Cf[i] = Cvt<T>::to_f(__ldg(gC + i));
                }
            }
            __syncwarp();
            mbar_wait(full, phase);
            phase ^= 1;
            char *orow = kOutF32 ? (char *)a.out + (((size_t)b * a.dim + d) * L + l0) * 4 : nullptr;
            // token loop, cut at the checkpoint boundaries so that its body is branch-free and can be software-pipelined
            for (int t0 = 0; t0 < len;) {
                const int nt = min(to_ck, len - t0);
#pragma unroll 7
                for (int t = t0; t < t0 + nt; t += 4) {
                    float2 dd[2], uu[2], Bv[2], Cv[2], y[2];
                    Quad<T>::ld(pd + t * es, dd);
                    Quad<T>::ld(pu + t * es, uu);
                    Quad<float>::ld(reinterpret_cast<const char *>(Bf + t), Bv);
                    Quad<float>::ld(reinterpret_cast<const char *>(Cf + t), Cv);
#pragma unroll
                    for (int q = 0; q < 2; ++q) {
                        float2 m = fma2(dd[q], kL2E, bl2);          // (delta + bias) * log2e
                        if (kSoftplus) {
                            const float2 e = make_float2(ex2f(fminf(m.x, 120.f)), ex2f(fminf(m.y, 120.f)));
                            const float2 sp = add2(e, kOne);
                            m = make_float2(fmaxf(lg2f(sp.x), m.x), fmaxf(lg2f(sp.y), m.y));   // softplus * log2e
                        }
                        msum = add2(msum, m);
                        const float2 arg = mul2(m, A2);
                        const float2 av = make_float2(ex2f(arg.x), ex2f(arg.y));
                        const float2 bv = mul2(mul2(m, uu[q]), Bv[q]);
                        float2 hh;
                        h = fmaf(av.x, h, bv.x); hh.x = h;
                        h = fmaf(av.y, h, bv.y); hh.y = h;
                        y[q] = fma2(hh, Cv[q], mul2(uu[q], D2));
                    }
                    if (kOutF32) *reinterpret_cast<float4 *>(orow + (size_t)t * 4) = make_float4(y[0].x, y[0].y, y[1].x, y[1].y);
                    else Quad<T>::st(pu + t * es, y);            // y replaces u in place
                }
                t0 += nt;
                to_ck -= nt;
                if (to_ck == 0) {
                    // checkpoint (prod a, h) at the boundaries shared with the warp-scan kernels and at the row end;
                    // prod a = 2^(A * sum m) -- one MUFU per checkpoint instead of one multiply per token
                    xrow[xc++] = make_float2(ex2f(Araw * (msum.x + msum.y)), h);
                    to_ck = min(a.xchunk_tokens, L - (l0 + t0));
                }
            }
            if (!kOutF32) {
                fence_proxy_async();
                __syncwarp();
                char *gout = (char *)a.out + (((size_t)b * a.dim + row0) * L + l0) * es;
                if (nch == 1) {
                    if (lane == 0) bulk_s2g(gout, tu, (uint32_t)(32 * L * es));
                } else {
                    bulk_s2g(gout + (size_t)lane * L * es, tu + (size_t)lane * Lc * es, (uint32_t)(len * es));
                }
                bulk_commit();
                bulk_wait_read<0>();                        // the tile is refilled next: it must have been read out
            }
            __syncwarp();
        }
    }
    asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");   // stores complete before the CTA retires
}

template <typename T>
cudaError_t launch_fwd_rows(const RowsArgs &a, int grid, bool out_f32, cudaStream_t stream) {
    void (*kernel)(const RowsArgs);
    if (a.softplus) kernel = out_f32 ? &ss_fwd_rows_kernel<T, true, true> : &ss_fwd_rows_kernel<T, true, false>;
    else kernel = out_f32 ? &ss_fwd_rows_kernel<T, false, true> : &ss_fwd_rows_kernel<T, false, false>;
    cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, a.smem_bytes);
    if (e != cudaSuccess) return e;
    kernel<<<grid, 32, a.smem_bytes, stream>>>(a);
    return cudaGetLastError();
}

}  // namespace mia
