// Forward selective scan, STREAMING row-serial path (d_state == 1): one LANE per row, tokens walked serially, the
// [32 rows x 32 tokens] pieces of u and delta streamed through a 2-stage cp.async ring private to the warp.
//
// Used for the shapes scan_fwd_rows.cuh cannot take: its tiles come from TMA bulk copies, which need 16-byte aligned
// pieces, and the rows of e.g. L = 260 bf16 tokens are 520 B apart, so every other row piece is only 8-byte aligned;
// 8-byte cp.async (LDGSTS) copies can move them.  Small stages (4.6 KB) also allow 16 warps per SM instead of 8, but
// that buys nothing: where both kernels apply they run at the same speed (72 us at M196; ncu: the forward is bound by
// the MIO queue -- MUFU plus shared-memory instructions -- not by occupancy, and LDGSTS / copy-out add to it), so the
// TMA kernel keeps precedence.  Structure, no block-wide state at all:
//   * lane (i, part) copies the 4-token piece `part` of rows 4 j + i (j = 0..7): a warp-level copy instruction moves 4
//     rows x 64 B; the shared-memory row pitch is padded by one piece so that the per-lane row reads are conflict-free;
//   * y overwrites u inside the stage and is copied out by the same (row, piece) mapping: 64-byte runs per row;
//   * B ln2 and C of the (batch, group) sit in shared memory as fp32 for the whole row (broadcast reads);
//   * (prod a, h) is checkpointed into x every 256 tokens (8 stages), like every other forward kernel.
// Any L % 4 == 0 works (long rows just take more stages).  Preconditions (host-checked): d_state == 1, delta per row,
// no z, rows contiguous (stride == L), rows_per_group % 32 == 0, u / delta / out aligned to one 4-token piece.
#pragma once
#include <type_traits>

#include "scan_fwd_rows.cuh"

namespace mia {

template <int kBytes> __device__ __forceinline__ void cp_async(void *sdst, const void *gsrc) {
    if (kBytes == 16) asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_u32(sdst)), "l"(gsrc) : "memory");
    else asm volatile("cp.async.ca.shared.global [%0], [%1], %2;" ::"r"(smem_u32(sdst)), "l"(gsrc), "n"(kBytes) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int kN> __device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(kN) : "memory"); }

template <typename T, bool kSoftplus, bool kOutF32>
__global__ void __launch_bounds__(32, 16) ss_fwd_stream_kernel(const __grid_constant__ StreamArgs a) {
    extern __shared__ __align__(128) char smem[];
    constexpr int es = (int)sizeof(T);
    constexpr int kPiece = 4 * es;                           // bytes of one 4-token piece (8 or 16)
    constexpr int kPitch = kStreamTok * es + kPiece;         // row pitch inside a stage (padded: conflict-free row reads)
    constexpr int kTile = 32 * kPitch;                       // one tensor of one stage
    const int lane = threadIdx.x;
    const int sub = lane >> 3, part = lane & 7;              // copy mapping: rows 4 j + sub, piece `part`
    float *Bf = reinterpret_cast<float *>(smem + a.off_bc32), *Cf = Bf + a.Lp;
    const int L = a.L;
    const int nst = (L + kStreamTok - 1) / kStreamTok;
    const int batches_per_group = a.rows_per_group / 32;
    const float *Ap = reinterpret_cast<const float *>(a.A);
    const float *Dp = reinterpret_cast<const float *>(a.D);
    const float *biasp = reinterpret_cast<const float *>(a.delta_bias);
    const float2 kL2E = splat2(kLog2e), kOne = splat2(1.f);
    using raw = typename Cvt<T>::raw;

    for (int item = blockIdx.x; item < a.n_items; item += gridDim.x) {
        const int bt = item % batches_per_group;
        const int bg = item / batches_per_group;
        const int g = bg % a.G, b = bg / a.G;
        const int row0 = g * a.rows_per_group + bt * 32;
        const int d = row0 + lane;
        const size_t goff = ((size_t)b * a.dim + row0) * L;
        const char *gu = (const char *)a.u + goff * es, *gd = (const char *)a.delta + goff * es;
        char *gout = (char *)a.out + goff * (kOutF32 ? 4 : es);

        auto issue = [&](int k) {                            // stage k -> buffer k & 1
            const int t0 = k * kStreamTok;
            const int npart = min(8, (L - t0) >> 2);
            char *su = smem + (k & 1) * 2 * kTile, *sd = su + kTile;
            if (part < npart) {
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    const int row = 4 * j + sub;
                    const size_t go = ((size_t)row * L + t0 + part * 4) * es;
                    cp_async<kPiece>(su + row * kPitch + part * kPiece, gu + go);
                    cp_async<kPiece>(sd + row * kPitch + part * kPiece, gd + go);
                }
            }
            cp_async_commit();
        };
        issue(0);
        if (nst > 1) issue(1);
        {   // B ln2, C rows of the (batch, group) as fp32; all loads of a lane in flight before the first store
            const raw *gB = reinterpret_cast<const raw *>(a.B) + (size_t)b * a.B_bs + (size_t)g * a.B_gs;
            const raw *gC = reinterpret_cast<const raw *>(a.C) + (size_t)b * a.C_bs + (size_t)g * a.C_gs;
            for (int base = 0; base < L; base += 32 * 8) {
                raw vb[8], vc[8];
#pragma unroll
                for (int k = 0; k < 8; ++k) {
                    const int i = min(base + k * 32 + lane, L - 1);
                    vb[k] = __ldg(gB + i);
                    vc[k] = __ldg(gC + i);
                }
#pragma unroll
                for (int k = 0; k < 8; ++k) {
                    const int i = base + k * 32 + lane;
                    if (i < L) { Bf[i] = Cvt<T>::to_f(vb[k]) * kLn2; Cf[i] = Cvt<T>::to_f(vc[k]); }
                }
            }
        }
        const float Araw = __ldg(Ap + d);
        const float Dv = Dp ? __ldg(Dp + d) : 0.f;
        const float2 bl2 = splat2((biasp ? __ldg(biasp + d) : 0.f) * kLog2e), A2 = splat2(Araw), D2 = splat2(Dv);
        float h = 0.f;
        float2 msum = make_float2(0.f, 0.f);
        float2 *xrow = reinterpret_cast<float2 *>(a.x) + ((size_t)b * a.dim + d) * a.xchunks;
        int xc = 0;

#pragma unroll 1
        for (int k = 0; k < nst; ++k) {
            if (k + 1 < nst) cp_async_wait<1>(); else cp_async_wait<0>();
            __syncwarp();                                    // pieces copied by the other lanes are visible
            const int t0 = k * kStreamTok;
            const int nq = min(8, (L - t0) >> 2);
            char *su = smem + (k & 1) * 2 * kTile;
            char *pu = su + lane * kPitch;
            const char *pd = su + kTile + lane * kPitch;
            char *orow = kOutF32 ? gout + ((size_t)lane * L + t0) * 4 : nullptr;
            auto quad = [&](int q) {
                float2 dd[2], uu[2], Bv[2], Cv[2], y[2];
                Quad<T>::ld(pd + q * kPiece, dd);
                Quad<T>::ld(pu + q * kPiece, uu);
                Quad<float>::ld(reinterpret_cast<const char *>(Bf + t0 + 4 * q), Bv);
                Quad<float>::ld(reinterpret_cast<const char *>(Cf + t0 + 4 * q), Cv);
#pragma unroll
                for (int p = 0; p < 2; ++p) {
                    float2 m = fma2(dd[p], kL2E, bl2);       // (delta + bias) * log2e
                    if (kSoftplus) {
                        const float2 e = make_float2(ex2f(fminf(m.x, 120.f)), ex2f(fminf(m.y, 120.f)));
                        const float2 sp = add2(e, kOne);
                        m = make_float2(fmaxf(lg2f(sp.x), m.x), fmaxf(lg2f(sp.y), m.y));   // softplus * log2e
                    }
                    msum = add2(msum, m);
                    const float2 arg = mul2(m, A2);
                    const float2 av = make_float2(ex2f(arg.x), ex2f(arg.y));
                    const float2 bv = mul2(mul2(m, uu[p]), Bv[p]);
                    float2 hh;
                    h = fmaf(av.x, h, bv.x); hh.x = h;
                    h = fmaf(av.y, h, bv.y); hh.y = h;
                    y[p] = fma2(hh, Cv[p], mul2(uu[p], D2));
                }
                if (kOutF32) *reinterpret_cast<float4 *>(orow + (size_t)q * 16) = make_float4(y[0].x, y[0].y, y[1].x, y[1].y);
                else Quad<T>::st(pu + q * kPiece, y);        // y replaces u in place
            };
            if (nq == 8) {
#pragma unroll
                for (int q = 0; q < 8; ++q) quad(q);
            } else {
#pragma unroll 1
                for (int q = 0; q < nq; ++q) quad(q);
            }
            if (((k + 1) & 7) == 0 || k == nst - 1)          // checkpoint every 256 tokens and at the row end
                xrow[xc++] = make_float2(ex2f(Araw * (msum.x + msum.y)), h);
            __syncwarp();
            if (!kOutF32 && part < nq) {                     // copy y out: (row, piece) mapping of the loads
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    const int row = 4 * j + sub;
                    const char *s = su + row * kPitch + part * kPiece;
                    char *gp = gout + ((size_t)row * L + t0 + part * 4) * es;
                    if (kPiece == 16) *reinterpret_cast<uint4 *>(gp) = *reinterpret_cast<const uint4 *>(s);
                    else *reinterpret_cast<uint2 *>(gp) = *reinterpret_cast<const uint2 *>(s);
                }
            }
            __syncwarp();                                    // the buffer is refilled next: everyone has read it
            if (k + 2 < nst) issue(k + 2);
        }
        __syncwarp();                                        // B' / C rows are rewritten by the next item
    }
}

template <typename T>
cudaError_t launch_fwd_stream(const StreamArgs &a, int grid, bool out_f32, cudaStream_t stream) {
    void (*kernel)(const StreamArgs);
    if (a.softplus) kernel = out_f32 ? &ss_fwd_stream_kernel<T, true, true> : &ss_fwd_stream_kernel<T, true, false>;
    else kernel = out_f32 ? &ss_fwd_stream_kernel<T, false, true> : &ss_fwd_stream_kernel<T, false, false>;
    cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, a.smem_bytes);
    if (e != cudaSuccess) return e;
    kernel<<<grid, 32, a.smem_bytes, stream>>>(a);
    return cudaGetLastError();
}

}  // namespace mia
