// Forward selective scan, ROW-SERIAL path for d_state = kN > 1 (SS2D's default d_state 16, the ARM / Vim mixers):
// one LANE per row, the kN states of the row live in registers, tokens are walked serially.
//
// Why: in the warp-scan formulation every state costs two 5-step shuffle scans plus per-state bookkeeping per 256-token
// warp pass (ncu, N = 16: 3200 executed warp-instructions per row, 4 % of them MUFU).  With a lane per row the
// recurrence is one packed FFMA2 per state PAIR and token, no shuffles, no idle lanes past the row end: ~5 instructions
// per state and token, and the kernel sits on the MUFU pipe (kN exponentials per row-token: exp(dl A_n) has no
// cheaper form for a free parameter A), which is the real ceiling of this configuration (DESIGN.md 3.4).
//   * u / delta tiles [32 rows x L]: one flat TMA bulk copy each; y overwrites u and leaves with one bulk store;
//   * a CTA is 4 warps, each with its own 32-row batch (own tiles, own mbarrier) of the same (batch, group); B and C of the
//     group are transposed once per group into token-major rows [t][kN] in shared memory (element type T: fp32 rows
//     would cost a resident CTA), so that every token needs kN/8 broadcast LDS.128 per tensor and one ALU op per value;
//   * log2 domain throughout: m = softplus(delta + bias) log2e, a_n = 2^(m A_n), b_n = (m u) (B_n ln2).
// With the z gate of the mamba_ssm signature the z tile is a third tile per warp (2 warps per CTA), out_z = y silu(z)
// overwrites it and leaves with a second bulk store; `out` (y before the gate) is still written: the backward needs it.
// Preconditions (host-checked, otherwise the warp-scan kernels run): d_state == kN, delta per row, whole rows in
// the tile (32 L es <= tile budget), rows contiguous, rows_per_group % 32 == 0, 16-byte aligned tiles; any L (odd L takes
// an element-wise path for u / delta / z / y inside the same kernel).
#pragma once
#include <type_traits>

#include "scan_fwd_rows.cuh"

namespace mia {

// kN states of one token, stored as T in shared memory (token-major), to kN/2 float2 state pairs.
template <typename T, int kN> struct StateRow;
template <int kN> struct StateRow<__nv_bfloat16, kN> {
    static __device__ __forceinline__ void ld(const void *p, float2 (&v)[kN / 2]) {
        const uint4 *q = reinterpret_cast<const uint4 *>(p);
#pragma unroll
        for (int i = 0; i < kN / 8; ++i) {
            const uint4 w = q[i];
            v[4 * i + 0] = make_float2(__uint_as_float(w.x << 16), __uint_as_float(w.x & 0xffff0000u));
            v[4 * i + 1] = make_float2(__uint_as_float(w.y << 16), __uint_as_float(w.y & 0xffff0000u));
            v[4 * i + 2] = make_float2(__uint_as_float(w.z << 16), __uint_as_float(w.z & 0xffff0000u));
            v[4 * i + 3] = make_float2(__uint_as_float(w.w << 16), __uint_as_float(w.w & 0xffff0000u));
        }
    }
};
template <int kN> struct StateRow<__half, kN> {
    static __device__ __forceinline__ void ld(const void *p, float2 (&v)[kN / 2]) {
        const uint4 *q = reinterpret_cast<const uint4 *>(p);
#pragma unroll
        for (int i = 0; i < kN / 8; ++i) {
            uint4 w = q[i];
            v[4 * i + 0] = __half22float2(*reinterpret_cast<__half2 *>(&w.x));
            v[4 * i + 1] = __half22float2(*reinterpret_cast<__half2 *>(&w.y));
            v[4 * i + 2] = __half22float2(*reinterpret_cast<__half2 *>(&w.z));
            v[4 * i + 3] = __half22float2(*reinterpret_cast<__half2 *>(&w.w));
        }
    }
};
template <int kN> struct StateRow<float, kN> {
    static __device__ __forceinline__ void ld(const void *p, float2 (&v)[kN / 2]) {
        const float4 *q = reinterpret_cast<const float4 *>(p);
#pragma unroll
        for (int i = 0; i < kN / 4; ++i) {
            const float4 w = q[i];
            v[2 * i] = make_float2(w.x, w.y);
            v[2 * i + 1] = make_float2(w.z, w.w);
        }
    }
};

template <typename T, bool kSoftplus, bool kOutF32, int kN, bool kHasZ>
__global__ void __launch_bounds__(32 * kRowsNWarps) ss_fwd_rowsn_kernel(const __grid_constant__ RowsNArgs a) {
    static_assert(kN % 8 == 0, "states are loaded eight at a time and processed as packed pairs");
    extern __shared__ __align__(128) char smem[];
    constexpr int es = (int)sizeof(T);
    constexpr int kP = kN / 2;
    using raw = typename Cvt<T>::raw;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int L = a.L;
    const int W = blockDim.x >> 5;
    char *tu = smem + (size_t)warp * a.tiles_per_warp * a.tile_bytes, *td = tu + a.tile_bytes, *tz = td + a.tile_bytes;
    raw *Bs = reinterpret_cast<raw *>(smem + a.off_bc), *Cs = Bs + (size_t)L * kN;     // [t][kN], element type T
    uint64_t *full = reinterpret_cast<uint64_t *>(smem + a.off_bar) + warp;
    if (lane == 0) { mbar_init(full, 1); fence_mbar_init(); }
    __syncthreads();

    const int batches_per_group = a.rows_per_group / 32;
    const float *Ap = reinterpret_cast<const float *>(a.A);
    const float *Dp = reinterpret_cast<const float *>(a.D);
    const float *biasp = reinterpret_cast<const float *>(a.delta_bias);
    const float2 kL2E = splat2(kLog2e), kOne = splat2(1.f);
    char *pu = tu + (size_t)lane * L * es;
    const char *pd = td + (size_t)lane * L * es;
    char *pz = tz + (size_t)lane * L * es;
    uint32_t phase = 0;

    // contiguous unit ranges per CTA (the first `rem` CTAs take one more): consecutive units share (batch, group), so the
    // B / C transposition below is redone only when the group changes
    const int q = a.n_units / gridDim.x, rem = a.n_units % gridDim.x;
    const int unit_begin = blockIdx.x * q + min((int)blockIdx.x, rem);
    const int unit_end = unit_begin + q + ((int)blockIdx.x < rem ? 1 : 0);
    int bg_loaded = -1;
    for (int unit = unit_begin; unit < unit_end; ++unit) {
        const int bg = unit / a.units_per_group;
        const int bt = (unit % a.units_per_group) * W + warp;
        const bool valid = bt < batches_per_group;       // warp-uniform
        const int g = bg % a.G, b = bg / a.G;
        const int row0 = g * a.rows_per_group + (valid ? bt : 0) * 32;
        const int d = row0 + lane;
        const size_t goff = ((size_t)b * a.dim + row0) * L;
        if (valid && lane == 0) {
            bulk_g2s(tu, (const char *)a.u + goff * es, (uint32_t)(32 * L * es), full);
            bulk_g2s(td, (const char *)a.delta + goff * es, (uint32_t)(32 * L * es), full);
            if (kHasZ) bulk_g2s(tz, (const char *)a.z + goff * es, (uint32_t)(32 * L * es), full);
            mbar_arrive_expect_tx(full, (kHasZ ? 3u : 2u) * 32u * L * es);
        }
        // B, C of the group: global [n][t] (sequence contiguous) -> shared [t][kN].  Flat index = t * kN + n: the shared
        // stores of a warp are consecutive elements, the global loads kN rows x 32 / kN tokens; 8 + 8 loads per thread
        // are in flight before the first store.
        if (bg != bg_loaded) {
            bg_loaded = bg;
            __syncthreads();                             // every warp is done with the previous group's rows
            const raw *gB = reinterpret_cast<const raw *>(a.B) + (size_t)b * a.B_bs + (size_t)g * a.B_gs;
            const raw *gC = reinterpret_cast<const raw *>(a.C) + (size_t)b * a.C_bs + (size_t)g * a.C_gs;
            constexpr int kU = 8;
            const int kStep = blockDim.x;
            const int tot = L * kN;
            for (int base = 0; base < tot; base += kStep * kU) {
                raw vb[kU], vc[kU];
#pragma unroll
                for (int k = 0; k < kU; ++k) {
                    const int idx = min(base + k * kStep + (int)threadIdx.x, tot - 1);
                    const int t = idx / kN, n = idx % kN;
                    vb[k] = __ldg(gB + (size_t)n * a.B_ns + t);
                    vc[k] = __ldg(gC + (size_t)n * a.C_ns + t);
                }
#pragma unroll
                for (int k = 0; k < kU; ++k) {
                    const int idx = base + k * kStep + (int)threadIdx.x;
                    if (idx < tot) { Bs[idx] = vb[k]; Cs[idx] = vc[k]; }
                }
            }
            __syncthreads();
        }
        if (!valid) continue;
        float2 A2[kP], h2[kP];
#pragma unroll
        for (int p = 0; p < kP; ++p) {
            A2[p] = make_float2(__ldg(Ap + (size_t)d * a.A_ds + (2 * p) * a.A_ns), __ldg(Ap + (size_t)d * a.A_ds + (2 * p + 1) * a.A_ns));
            h2[p] = make_float2(0.f, 0.f);
        }
        const float Dv = Dp ? __ldg(Dp + d) : 0.f;
        const float2 bl2 = splat2((biasp ? __ldg(biasp + d) : 0.f) * kLog2e);
        float msum = 0.f;
        mbar_wait(full, phase);
        phase ^= 1;
        char *orow = kOutF32 ? (char *)a.out + (goff + (size_t)lane * L) * 4 : nullptr;
        char *ozrow = (kOutF32 && kHasZ) ? (char *)a.out_z + (goff + (size_t)lane * L) * 4 : nullptr;

        // one token of this lane's row: all kN states advance, returns y (before the gate)
        auto token = [&](const float m, const float uval, const int t) -> float {
            const float2 m2 = splat2(m), mu2 = splat2(m * uval * kLn2);                // dl u = m u ln2
            msum += m;
            float2 Bv[kP], Cv[kP];
            StateRow<T, kN>::ld(Bs + (size_t)t * kN, Bv);
            StateRow<T, kN>::ld(Cs + (size_t)t * kN, Cv);
            float2 yacc = make_float2(0.f, 0.f);
#pragma unroll
            for (int p = 0; p < kP; ++p) {
                const float2 arg = mul2(m2, A2[p]);
                const float2 av = make_float2(ex2f(arg.x), ex2f(arg.y));
                h2[p] = fma2(av, h2[p], mul2(mu2, Bv[p]));
                yacc = fma2(h2[p], Cv[p], yacc);
            }
            return fmaf(Dv, uval, yacc.x + yacc.y);
        };
        if ((L & 3) == 0) {
#pragma unroll 1
            for (int t = 0; t < L; t += 4) {
                float2 dd[2], uu[2], y[2];
                Quad<T>::ld(pd + t * es, dd);
                Quad<T>::ld(pu + t * es, uu);
                float mm[4], us[4] = {uu[0].x, uu[0].y, uu[1].x, uu[1].y}, ys[4];
#pragma unroll
                for (int qq = 0; qq < 2; ++qq) {
                    float2 m = fma2(dd[qq], kL2E, bl2);         // (delta + bias) * log2e
                    if (kSoftplus) {
                        const float2 e = make_float2(ex2f(fminf(m.x, 120.f)), ex2f(fminf(m.y, 120.f)));
                        const float2 sp = add2(e, kOne);
                        m = make_float2(fmaxf(lg2f(sp.x), m.x), fmaxf(lg2f(sp.y), m.y));   // softplus * log2e
                    }
                    mm[2 * qq] = m.x; mm[2 * qq + 1] = m.y;
                }
#pragma unroll
                for (int i = 0; i < 4; ++i) ys[i] = token(mm[i], us[i], t + i);
                y[0] = make_float2(ys[0], ys[1]);
                y[1] = make_float2(ys[2], ys[3]);
                if (kOutF32) *reinterpret_cast<float4 *>(orow + (size_t)t * 4) = make_float4(ys[0], ys[1], ys[2], ys[3]);
                else Quad<T>::st(pu + t * es, y);                // y replaces u in place
                if (kHasZ) {                                     // out_z = y * silu(z), computed from the unrounded y
                    float2 zz[2], yz[2];
                    Quad<T>::ld(pz + t * es, zz);
#pragma unroll
                    for (int qq = 0; qq < 2; ++qq) {
                        const float2 sz = make_float2(rcpf(1.f + ex2f(-zz[qq].x * kLog2e)), rcpf(1.f + ex2f(-zz[qq].y * kLog2e)));
                        yz[qq] = mul2(mul2(y[qq], zz[qq]), sz);
                    }
                    if (kOutF32) *reinterpret_cast<float4 *>(ozrow + (size_t)t * 4) = make_float4(yz[0].x, yz[0].y, yz[1].x, yz[1].y);
                    else Quad<T>::st(pz + t * es, yz);           // out_z replaces z in place
                }
            }
        } else {
            // odd lengths (L = 197 with the cls token of the ARM encoders): rows of the tile are only element-aligned, so u,
            // delta, z and y move one element at a time -- two or three extra shared-memory instructions on ~100 per token
#pragma unroll 1
            for (int t = 0; t < L; ++t) {
                const float dl = Cvt<T>::to_f(*reinterpret_cast<const raw *>(pd + t * es));
                const float uval = Cvt<T>::to_f(*reinterpret_cast<const raw *>(pu + t * es));
                float m = fmaf(dl, kLog2e, bl2.x);
                if (kSoftplus) m = fmaxf(lg2f(1.f + ex2f(fminf(m, 120.f))), m);
                const float yv = token(m, uval, t);
                if (kOutF32) *reinterpret_cast<float *>(orow + (size_t)t * 4) = yv;
                else *reinterpret_cast<raw *>(pu + t * es) = Cvt<T>::from_f(yv);
                if (kHasZ) {
                    const float zv = Cvt<T>::to_f(*reinterpret_cast<const raw *>(pz + t * es));
                    const float yz = yv * zv * rcpf(1.f + ex2f(-zv * kLog2e));
                    if (kOutF32) *reinterpret_cast<float *>(ozrow + (size_t)t * 4) = yz;
                    else *reinterpret_cast<raw *>(pz + t * es) = Cvt<T>::from_f(yz);
                }
            }
        }
        // checkpoint at the row end: (prod a_n, h_n) interleaved, prod a_n = 2^(A_n sum m)
        {
            float4 *xr = reinterpret_cast<float4 *>(a.x + ((size_t)b * a.dim + d) * (2 * kN));
#pragma unroll
            for (int p = 0; p < kP; ++p)
                xr[p] = make_float4(ex2f(A2[p].x * msum), h2[p].x, ex2f(A2[p].y * msum), h2[p].y);
        }
        if (!kOutF32) {
            fence_proxy_async();
            __syncwarp();
            if (lane == 0) {
                bulk_s2g((char *)a.out + goff * es, tu, (uint32_t)(32 * L * es));
                if (kHasZ) bulk_s2g((char *)a.out_z + goff * es, tz, (uint32_t)(32 * L * es));
                bulk_commit();
                bulk_wait_read<0>();                        // the tile is refilled next: it must have been read out
            }
        }
        __syncwarp();
    }
    asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");   // stores complete before the CTA retires
}

template <typename T, int kN, bool kHasZ>
void (*pick_fwd_rowsn(bool softplus, bool out_f32))(const RowsNArgs) {
    if (softplus) return out_f32 ? &ss_fwd_rowsn_kernel<T, true, true, kN, kHasZ> : &ss_fwd_rowsn_kernel<T, true, false, kN, kHasZ>;
    return out_f32 ? &ss_fwd_rowsn_kernel<T, false, true, kN, kHasZ> : &ss_fwd_rowsn_kernel<T, false, false, kN, kHasZ>;
}

template <typename T>
cudaError_t launch_fwd_rowsn(const RowsNArgs &a, int grid, bool out_f32, cudaStream_t stream) {
    void (*kernel)(const RowsNArgs) = nullptr;
    const bool sp = a.softplus != 0, hz = a.z != nullptr;
    if (a.N == 16) kernel = hz ? pick_fwd_rowsn<T, 16, true>(sp, out_f32) : pick_fwd_rowsn<T, 16, false>(sp, out_f32);
    else if (a.N == 8) kernel = hz ? pick_fwd_rowsn<T, 8, true>(sp, out_f32) : pick_fwd_rowsn<T, 8, false>(sp, out_f32);
    else return cudaErrorInvalidValue;
    cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, a.smem_bytes);
    if (e != cudaSuccess) return e;
    kernel<<<grid, 32 * a.warps, a.smem_bytes, stream>>>(a);
    return cudaGetLastError();
}

}  // namespace mia
