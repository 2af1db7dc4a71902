// Forward selective scan for LONG rows and FEW of them (d_state == 1), e.g. L = 6400 at batch 4: chunk-parallel.
//
// The row-serial kernel (scan_fwd_rows.cuh) walks a row from its first to its last token inside one warp; with 4 x 3072
// rows there are only 384 such warps for 148 SMs (2.6 per SM) and each is latency-bound for 6400 tokens.  The recurrence
// h = a h + b is associative, so the row is cut at the 256-token checkpoint boundaries of x and done in three launches:
//   A  per (32-row batch, chunk): local scan from h = 0, only the aggregate (P = prod a, h_local) is kept -> x[b][d][c];
//   B  per row: the chunk aggregates are chained serially, x[b][d][c] <- (prod a so far, state after chunk c)   (nch steps);
//   C  per (32-row batch, chunk): the real pass, starting from the state after chunk c - 1, writes the outputs.
// 1.6x the arithmetic of the serial kernel (pass A needs the same 3 MUFU per token), but 25x the parallelism at L = 6400;
// u and delta are read twice (the kernels are not HBM-bound).  x is exactly what the serial kernels would have written,
// so any backward kernel can consume it.  Lane per row, one-warp CTAs, per-row TMA pieces with a padded pitch, y in place
// + bulk stores, log2-domain arithmetic: as in scan_fwd_rows.cuh.
// Preconditions (host-checked): d_state == 1, delta per row, no z, rows contiguous and 16-byte aligned pieces
// (L es % 16 == 0), rows_per_group % 32 == 0, L % 4 == 0, more than one 256-token chunk.
#pragma once
#include <type_traits>

#include "scan_fwd_rows.cuh"

namespace mia {

template <typename T, bool kSoftplus, bool kOutF32, bool kStateOnly>
__global__ void __launch_bounds__(32) ss_fwd_chunk_kernel(const __grid_constant__ ChunkArgs a) {
    extern __shared__ __align__(128) char smem[];
    constexpr int es = (int)sizeof(T);
    constexpr int kPitch = kChunkTok * es + 16;              // a 512-byte pitch would put all lanes on the same banks
    const int lane = threadIdx.x;
    char *tu = smem, *td = smem + a.tile_bytes;
    float *Bf = reinterpret_cast<float *>(smem + a.off_bc32), *Cf = Bf + kChunkTok;
    uint64_t *full = reinterpret_cast<uint64_t *>(smem + a.off_bar);
    if (lane == 0) { mbar_init(full, 1); fence_mbar_init(); }
    __syncwarp();

    const int L = a.L, nch = a.n_chunks;
    const int batches_per_group = a.rows_per_group / 32;
    const float *Ap = reinterpret_cast<const float *>(a.A);
    const float *Dp = reinterpret_cast<const float *>(a.D);
    const float *biasp = reinterpret_cast<const float *>(a.delta_bias);
    const float2 kL2E = splat2(kLog2e), kOne = splat2(1.f);
    char *pu = tu + (size_t)lane * kPitch;
    const char *pd = td + (size_t)lane * kPitch;
    uint32_t phase = 0;
    using raw = typename Cvt<T>::raw;

    for (int item = blockIdx.x; item < a.n_items; item += gridDim.x) {
        const int c = item % nch, rb = item / nch;           // chunk-fastest: neighbouring CTAs touch neighbouring memory
        const int bt = rb % batches_per_group;
        const int bg = rb / batches_per_group;
        const int g = bg % a.G, b = bg / a.G;
        const int row0 = g * a.rows_per_group + bt * 32;
        const int d = row0 + lane;
        const int l0 = c * kChunkTok, len = min(kChunkTok, L - l0);
        const size_t gro = ((size_t)b * a.dim + d) * L + l0;  // this lane's row piece
        bulk_g2s(pu, (const char *)a.u + gro * es, (uint32_t)(len * es), full);
        bulk_g2s(const_cast<char *>(pd), (const char *)a.delta + gro * es, (uint32_t)(len * es), full);
        __syncwarp();
        if (lane == 0) mbar_arrive_expect_tx(full, 64u * len * es);
        {
            const raw *gB = reinterpret_cast<const raw *>(a.B) + (size_t)b * a.B_bs + (size_t)g * a.B_gs + l0;
            const raw *gC = reinterpret_cast<const raw *>(a.C) + (size_t)b * a.C_bs + (size_t)g * a.C_gs + l0;
            raw vb[8], vc[8];
#pragma unroll
            for (int k = 0; k < 8; ++k) {
                const int i = min(k * 32 + lane, len - 1);
                vb[k] = __ldg(gB + i);
                if (!kStateOnly) vc[k] = __ldg(gC + i);
            }
#pragma unroll
            for (int k = 0; k < 8; ++k) {
                const int i = k * 32 + lane;
                Bf[i] = i < len ? Cvt<T>::to_f(vb[k]) * kLn2 : 0.f;
                if (!kStateOnly) Cf[i] = i < len ? Cvt<T>::to_f(vc[k]) : 0.f;
            }
        }
        const float Araw = __ldg(Ap + d);
        const float Dv = (!kStateOnly && Dp) ? __ldg(Dp + d) : 0.f;
        const float2 bl2 = splat2((biasp ? __ldg(biasp + d) : 0.f) * kLog2e), A2 = splat2(Araw), D2 = splat2(Dv);
        float2 *xrow = reinterpret_cast<float2 *>(a.x) + ((size_t)b * a.dim + d) * nch;
        float h = (!kStateOnly && c > 0) ? xrow[c - 1].y : 0.f;
        float2 msum = make_float2(0.f, 0.f);
        __syncwarp();
        mbar_wait(full, phase);
        phase ^= 1;
        char *orow = (kOutF32 && !kStateOnly) ? (char *)a.out + gro * 4 : nullptr;
#pragma unroll 4
        for (int t = 0; t < len; t += 4) {
            float2 dd[2], uu[2], Bv[2], Cv[2], y[2];
            Quad<T>::ld(pd + t * es, dd);
            Quad<T>::ld(pu + t * es, uu);
            Quad<float>::ld(reinterpret_cast<const char *>(Bf + t), Bv);
            if (!kStateOnly) Quad<float>::ld(reinterpret_cast<const char *>(Cf + t), Cv);
#pragma unroll
            for (int q = 0; q < 2; ++q) {
                float2 m = fma2(dd[q], kL2E, bl2);           // (delta + bias) * log2e
                if (kSoftplus) {
                    const float2 e = make_float2(ex2f(fminf(m.x, 120.f)), ex2f(fminf(m.y, 120.f)));
                    const float2 sp = add2(e, kOne);
                    m = make_float2(fmaxf(lg2f(sp.x), m.x), fmaxf(lg2f(sp.y), m.y));   // softplus * log2e
                }
                if (kStateOnly) msum = add2(msum, m);
                const float2 arg = mul2(m, A2);
                const float2 av = make_float2(ex2f(arg.x), ex2f(arg.y));
                const float2 bv = mul2(mul2(m, uu[q]), Bv[q]);
                float2 hh;
                h = fmaf(av.x, h, bv.x); hh.x = h;
                h = fmaf(av.y, h, bv.y); hh.y = h;
                if (!kStateOnly) y[q] = fma2(hh, Cv[q], mul2(uu[q], D2));
            }
            if (!kStateOnly) {
                if (kOutF32) *reinterpret_cast<float4 *>(orow + (size_t)t * 4) = make_float4(y[0].x, y[0].y, y[1].x, y[1].y);
                else Quad<T>::st(pu + t * es, y);            // y replaces u in place
            }
        }
        if (kStateOnly) {
            xrow[c] = make_float2(ex2f(Araw * (msum.x + msum.y)), h);   // (prod a, local end state) of the chunk
        } else if (!kOutF32) {
            fence_proxy_async();
            __syncwarp();
            bulk_s2g((char *)a.out + gro * es, pu, (uint32_t)(len * es));
            bulk_commit();
            bulk_wait_read<0>();                             // the tile is refilled next: it must have been read out
        }
        __syncwarp();
    }
    asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
}

// pass B: chain the chunk aggregates of every row; x[row][c] <- (prod a from the row start, state after chunk c): the same
// running prefix the serial kernels (and the reference, fwd_kernel_oflex.cuh:156-166) leave in x
template <typename T>   // (template only so that the header can live in several translation units)
__global__ void __launch_bounds__(256) ss_fwd_chunk_combine_kernel(float2 *x, const int n_rows, const int nch) {
    const int row = blockIdx.x * blockDim.x + threadIdx.x;
    if (row >= n_rows) return;
    float2 *xr = x + (size_t)row * nch;
    float h = 0.f, P = 1.f;
    for (int c = 0; c < nch; ++c) {
        const float2 v = xr[c];
        h = fmaf(v.x, h, v.y);
        P *= v.x;
        xr[c] = make_float2(P, h);
    }
}

template <typename T>
cudaError_t launch_fwd_chunks(const ChunkArgs &a, int grid, bool out_f32, cudaStream_t stream) {
    void (*ka)(const ChunkArgs) = a.softplus ? &ss_fwd_chunk_kernel<T, true, false, true> : &ss_fwd_chunk_kernel<T, false, false, true>;
    void (*kc)(const ChunkArgs);
    if (a.softplus) kc = out_f32 ? &ss_fwd_chunk_kernel<T, true, true, false> : &ss_fwd_chunk_kernel<T, true, false, false>;
    else kc = out_f32 ? &ss_fwd_chunk_kernel<T, false, true, false> : &ss_fwd_chunk_kernel<T, false, false, false>;
    cudaError_t e = cudaFuncSetAttribute(ka, cudaFuncAttributeMaxDynamicSharedMemorySize, a.smem_bytes);
    if (e != cudaSuccess) return e;
    e = cudaFuncSetAttribute(kc, cudaFuncAttributeMaxDynamicSharedMemorySize, a.smem_bytes);
    if (e != cudaSuccess) return e;
    ka<<<grid, 32, a.smem_bytes, stream>>>(a);
    const int n_rows = a.batch * a.dim;
    ss_fwd_chunk_combine_kernel<T><<<(n_rows + 255) / 256, 256, 0, stream>>>(reinterpret_cast<float2 *>(a.x), n_rows, a.n_chunks);
    kc<<<grid, 32, a.smem_bytes, stream>>>(a);
    return cudaGetLastError();
}

}  // namespace mia
