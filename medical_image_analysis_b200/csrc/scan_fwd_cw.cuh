// Forward selective scan, COLUMN-WALK row-serial path (d_state == 1): one lane per row, tokens walked serially, the data
// moved by 2-D tensor-map TMA boxes (cp.async.bulk.tensor.2d, SASS UTMALDG / UTMASTG) through a ring of small stages.
//
// What it fixes relative to scan_fwd_rows.cuh (measured, gpurun r2f): that kernel stages [32 rows x 200 tokens] chunks in ONE
// buffer (load, wait, compute, store, wait) with 8 warps per SM, so every chunk exposes a full load latency, and with 13 KB
// tiles 1536 work items fall 1.3 to a CTA (L = 6400, B = 16: 34 % of the HBM roofline against 57 % at L = 196).  Here
//   * a warp owns 32 tensor-map rows and walks them in windows of 32 columns; a window of u and of delta is one box copy each
//     (2 KB for 2-byte types), issued by lane 0 into a ring of 3-4 stages, two or three windows ahead of the one being
//     computed; completion is an mbarrier per stage;
//   * y replaces u in the stage and leaves with one box store; the stage is refilled one step later, when
//     cp.async.bulk.wait_group.read says the store has been read out -- no step waits for its own store;
//   * 12-16 KB of shared memory per warp: 13-16 resident warps per SM, and a B = 16, L = 6400 problem (1536 items) is
//     resident all at once instead of 1.3 rounds;
//   * tiles carry the TMA swizzle whose span is the tile row (64 B -> SWIZZLE_64B, 128 B -> SWIZZLE_128B): the 32 lanes read
//     the same column of 32 different rows, which unswizzled would hit 2-4 banks.
// Rows whose byte pitch is not a multiple of 16 (L = 196 bf16: 392 B) cannot be a tensor-map row; g = 2 or 4 consecutive rows
// can.  The tensor is then mapped as [rows / g][g L] and a lane walks its g rows one after the other (columns [s L, (s + 1) L)
// are row s) as one sequence, resetting the state at every multiple of L.  Box starts stay multiples of 32 columns, i.e.
// 16-byte aligned (a box starting at an odd row's first token would not be, and the TMA unit traps on it).  g is the smallest
// of 1, 2, 4 that makes the tensor-map row a multiple of 32 BYTES (L = 196 bf16: g = 4, 1568 B): with a 784-byte pitch every
// second tensor-map row starts in the middle of a 32-byte sector, each 64-byte box row then touches three sectors, and the
// forward read 19 % more DRAM bytes than it needed (ncu, profiles/r2z_ncu_summary.json).
//
// Block states for the backward (hblk): the state entering every 16-COLUMN group, slot j = column / 16, layout
// [item][ngrp][32 lanes].  For g = 1 that is the state entering token 16 j; for g = 2 the odd row's slots sit at tokens
// 16 j - L (its groups are aligned to columns, not to its own tokens) -- the layout scan_bwd_cw.cuh walks.
// Preconditions (host-checked): d_state == 1, delta per row, no z, dense rows, rows_per_group % (32 g) == 0, L % 4 == 0,
// 16-byte aligned tensors.
#pragma once
#include <cuda.h>

#include <type_traits>

#include "scan_fwd_rows.cuh"

namespace mia {

#ifndef MIA_CW_OCT
#define MIA_CW_OCT 1             // 0: the 8-byte (quad) tile accesses of the first version, kept for A/B timing (tools/ab_cw.py)
#endif

// Per-lane view of its row inside a [32 rows][RB bytes] tile written by TMA (tile base 1024-byte aligned) with the swizzle whose
// span equals the row: RB = 64 -> CU_TENSOR_MAP_SWIZZLE_64B (16-byte chunk index ^= address bits 7-8), RB = 128 -> SWIZZLE_128B
// (chunk index ^= address bits 7-9).  Byte b of the row sits at line + ((b & ~15) ^ y) + (b & 15).
struct SwzRow {
    uint32_t line, y;
    __device__ __forceinline__ uint32_t at(uint32_t b) const { return line + ((b & ~15u) ^ y) + (b & 15u); }
};
template <int RB>
__device__ __forceinline__ SwzRow swz_row(int row) {
    static_assert(RB == 64 || RB == 128, "tile rows of 64 or 128 bytes");
    const uint32_t off = (uint32_t)(row * RB);
    SwzRow r;
    r.line = off & ~127u;
    r.y = (off & 127u) ^ (((off >> 7) & (RB == 64 ? 3u : 7u)) << 4);
    return r;
}

__device__ __forceinline__ void tma_box_g2s(void *smem_dst, const CUtensorMap *tm, int c0, int c1, uint64_t *bar) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(smem_u32(smem_dst)),
                 "l"(tm), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
                 : "memory");
}
__device__ __forceinline__ void tma_box_s2g(const CUtensorMap *tm, const void *smem_src, int c0, int c1) {
    asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(tm), "r"(smem_u32(smem_src)), "r"(c0), "r"(c1)
                 : "memory");
}

template <typename T, bool kSoftplus, bool kOutF32, int kG>
__global__ void __launch_bounds__(32, 16) ss_fwd_cw_kernel(const __grid_constant__ CUtensorMap tm_u, const __grid_constant__ CUtensorMap tm_d,
                                                           const __grid_constant__ CUtensorMap tm_y, const __grid_constant__ CwFwdArgs a) {
    // The swizzled tiles need 1024-byte alignment.  The dynamic shared memory of a kernel without static shared memory starts at
    // the CTA's shared window, which is allocated in 1 KB units: asserted once instead of re-aligned at run time.
    extern __shared__ __align__(1024) char smem[];
    if ((smem_u32(smem) & 1023u) != 0) __trap();
    constexpr int es = (int)sizeof(T);
    constexpr int eo = kOutF32 ? 4 : es;
    using TO = typename std::conditional<kOutF32, float, T>::type;
    using raw = typename Cvt<T>::raw;
    constexpr int RBi = kCwTok * es, RBo = kCwTok * eo;
    constexpr int kTileI = 32 * RBi, kTileO = 32 * RBo;
    constexpr bool kOct = es == 2 && MIA_CW_OCT;                         // 16-byte tile accesses (8 tokens) for 2-byte types
    const int lane = threadIdx.x;
    float *Bw = reinterpret_cast<float *>(smem + a.off_bc32), *Cw = Bw + kCwTok;
    uint64_t *full = reinterpret_cast<uint64_t *>(smem + a.off_bar);
    const int ns = a.ns;
    if (lane == 0) {
        for (int s = 0; s < ns; ++s) mbar_init(full + s, 1);
        fence_mbar_init();
    }
    __syncwarp();
    const int L = a.L, ncols = kG * L, nwin = a.nwin;
    const int rows_per_item = 32 * kG;
    const int items_per_group = a.rows_per_group / rows_per_item;
    const float *Ap = reinterpret_cast<const float *>(a.A);
    const float *Dp = reinterpret_cast<const float *>(a.D);
    const float *biasp = reinterpret_cast<const float *>(a.delta_bias);
    const float2 kL2E = splat2(kLog2e), kOne = splat2(1.f);
    const SwzRow ri = swz_row<RBi>(lane), ro = swz_row<RBo>(lane);

    // A / D loads are consumed where they are issued, by a value-preserving ALU op that ptxas cannot remove (a.zero is 0 at run
    // time).  Otherwise their first use sits in the window loop and carries a wait on the scoreboard slot of these loads - the slot
    // the loop's own B / C prefetch loads use too, so EVERY window waited for the prefetch it had just issued instead of one window
    // later (ncu r2zz, profiles/README.md: 22 % of the warp samples of the L = 6400 forward on that one FMUL2, 11 % on one branch at
    // L = 196; the wait masks: tools/sass_waits.py).
    auto settle = [&](const float v) { return __uint_as_float(__float_as_uint(v) ^ (uint32_t)a.zero); };

    // first tensor-map row of an item, and its (batch, group) pair
    auto item_rows = [&](int item, int &b, int &gq, int &row0) {
        const int bt = item % items_per_group;
        const int bg = item / items_per_group;
        gq = bg % a.G; b = bg / a.G;
        row0 = gq * a.rows_per_group + bt * rows_per_item;
    };

    // ---- load stream: (item, window) pairs in the order this CTA computes them, `ns - 1` windows ahead
    int ld_item = blockIdx.x, ld_w = 0, ld_srow0 = 0, ld_stage = 0;
    if (ld_item < a.n_items) { int b, gq, r0; item_rows(ld_item, b, gq, r0); ld_srow0 = (b * a.dim + r0) / kG; }
    auto issue_load = [&]() {                                           // lane 0 only; no-op past the last item
        if (ld_item < a.n_items) {
            char *st = smem + ld_stage * a.stage_bytes;
            mbar_arrive_expect_tx(full + ld_stage, 2u * kTileI);
            tma_box_g2s(st, &tm_u, ld_w * kCwTok, ld_srow0, full + ld_stage);
            tma_box_g2s(st + kTileI, &tm_d, ld_w * kCwTok, ld_srow0, full + ld_stage);
            if (++ld_w == nwin) {
                ld_w = 0;
                ld_item += gridDim.x;
                if (ld_item < a.n_items) { int b, gq, r0; item_rows(ld_item, b, gq, r0); ld_srow0 = (b * a.dim + r0) / kG; }
            }
        }
        ld_stage = ld_stage + 1 == ns ? 0 : ld_stage + 1;
    };
    if (lane == 0)
        for (int s = 0; s < ns - 1; ++s) issue_load();

    uint32_t phbits = 0;                                                 // bit s: parity to wait for on full[s]
    int stage = 0, nstore = 0;
    // B / C of the window about to be computed, prefetched one window ahead into registers
    raw bnext = 0, cnext = 0;
    const raw *gB = nullptr, *gC = nullptr;                              // B / C rows of the item the prefetch is in
    auto bc_rows = [&](int item) {
        if (item < a.n_items) {
            int b, gq, r0;
            item_rows(item, b, gq, r0);
            gB = reinterpret_cast<const raw *>(a.B) + (size_t)b * a.B_bs + (size_t)gq * a.B_gs;
            gC = reinterpret_cast<const raw *>(a.C) + (size_t)b * a.C_bs + (size_t)gq * a.C_gs;
        } else {
            gB = gC = nullptr;
        }
    };
    auto fetch_bc = [&](int w) {
        const int c = w * kCwTok + lane;
        int tk = c;                                                      // token of column c: c mod L
#pragma unroll
        for (int i = 1; i < kG; ++i) tk -= tk >= L ? L : 0;
        const bool ok = gB != nullptr && c < ncols;
        bnext = ok ? __ldg(gB + tk) : (raw)0;
        cnext = ok ? __ldg(gC + tk) : (raw)0;
    };
    bc_rows(blockIdx.x);
    fetch_bc(0);

    for (int item = blockIdx.x; item < a.n_items; item += gridDim.x) {
        int b, gq, row0;
        item_rows(item, b, gq, row0);
        const int srow0 = (b * a.dim + row0) / kG;
        int seg = 0;                                                     // row of the tensor-map row being walked
        int d = row0 + kG * lane;
        float Araw = settle(__ldg(Ap + d));
        float2 bl2 = splat2((biasp ? __ldg(biasp + d) : 0.f) * kLog2e), A2 = splat2(Araw), D2 = splat2(settle(Dp ? __ldg(Dp + d) : 0.f));
        float h = 0.f;
        float2 msum = make_float2(0.f, 0.f);
        float2 *xrow = reinterpret_cast<float2 *>(a.x) + ((size_t)b * a.dim + d) * a.xchunks;
        int xc = 0;
        float *hb = a.hblk ? a.hblk + (size_t)item * a.ngrp * 32 + lane : nullptr;

        for (int w = 0; w < nwin; ++w) {
            const int c0 = w * kCwTok;
            Bw[lane] = Cvt<T>::to_f(bnext) * kLn2;                       // B' = B ln2, C as fp32 (zero past the end)
            Cw[lane] = Cvt<T>::to_f(cnext);
            if (w + 1 < nwin) {
                fetch_bc(w + 1);
            } else {
                bc_rows(item + gridDim.x);
                fetch_bc(0);
            }
            __syncwarp();
            mbar_wait(full + stage, (phbits >> stage) & 1u);
            phbits ^= 1u << stage;
            char *tu = smem + stage * a.stage_bytes;
            const char *td = tu + kTileI;
            char *ty = kOutF32 ? smem + a.off_out + (nstore & 1) * kTileO : tu;

            // columns [ca, cb) of the window, all of one row
            auto run = [&](const int ca, const int cb) {
                // kNQ quads = 4 kNQ tokens from column c on: one quad, or (2-byte types) two quads = one 16-byte access per tile
                // and lane -- conflict-free on the swizzled tile where 8-byte accesses are not (Oct, scan_fwd_rows.cuh)
                auto span = [&](const int c, auto nq_tag) {
                    constexpr int kNQ = decltype(nq_tag)::value, kNP = 2 * kNQ;
                    const int lc = c - c0;
                    float2 dd[kNP], uu[kNP], Bv[kNP], Cv[kNP], y[kNP];
                    if constexpr (kNQ == 2) {
                        Oct<T>::ld(td + ri.at(lc * es), dd);
                        Oct<T>::ld(tu + ri.at(lc * es), uu);
                    } else {
                        Quad<T>::ld(td + ri.at(lc * es), dd);
                        Quad<T>::ld(tu + ri.at(lc * es), uu);
                    }
#pragma unroll
                    for (int j = 0; j < kNQ; ++j) {
                        Quad<float>::ld(reinterpret_cast<const char *>(Bw + lc + 4 * j), *reinterpret_cast<float2(*)[2]>(&Bv[2 * j]));
                        Quad<float>::ld(reinterpret_cast<const char *>(Cw + lc + 4 * j), *reinterpret_cast<float2(*)[2]>(&Cv[2 * j]));
                    }
#pragma unroll
                    for (int q = 0; q < kNP; ++q) {
                        float2 m = fma2(dd[q], kL2E, bl2);              // (delta + bias) * log2e
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
                    if constexpr (kOutF32) {
#pragma unroll
                        for (int j = 0; j < kNQ; ++j) Quad<float>::st(ty + ro.at((lc + 4 * j) * 4), *reinterpret_cast<float2(*)[2]>(&y[2 * j]));
                    } else if constexpr (kNQ == 2) {
                        Oct<T>::st(tu + ri.at(lc * es), y);             // y replaces u in place
                    } else {
                        Quad<T>::st(tu + ri.at(lc * es), y);
                    }
                    // state entering the next 16-column group (coalesced: 32 lanes x 4 bytes)
                    const int ce = c + 4 * kNQ;
                    if (hb && (ce & 15) == 0 && ce < ncols) hb[(ce >> 4) * 32] = h;
                };
                using One = std::integral_constant<int, 1>;
                using Two = std::integral_constant<int, 2>;
                if constexpr (kOct) {
                    if (cb - ca == kCwTok) {
#pragma unroll
                        for (int q = 0; q < kCwTok / 8; ++q) span(ca + 8 * q, Two{});
                    } else {                                             // (row ends are multiples of 4 columns, not of 8)
                        int c = ca;
                        if ((c & 4) && c < cb) { span(c, One{}); c += 4; }
                        for (; c + 8 <= cb; c += 8) span(c, Two{});
                        if (c < cb) span(c, One{});
                    }
                } else {
                    if (cb - ca == kCwTok) {
#pragma unroll
                        for (int q = 0; q < kCwTok / 4; ++q) span(ca + 4 * q, One{});
                    } else {
                        for (int c = ca; c < cb; c += 4) span(c, One{});
                    }
                }
            };
            // checkpoint (cumulative prod a, h) of the current row: at the chunk boundaries shared with the warp-scan kernels
            // (multiples of 32 tokens) and at the row end
            auto checkpoint = [&](const int tok_end) {
                if (tok_end == L || (tok_end & (a.xchunk_tokens - 1)) == 0) xrow[xc++] = make_float2(ex2f(Araw * (msum.x + msum.y)), h);
            };
            const int cend = min(c0 + kCwTok, ncols);
            if (kG == 1) {
                run(c0, cend);
                checkpoint(cend);
            } else {
                // the window may hold the end of one row and the start of the next (several, for rows shorter than a window)
                int c = c0;
                while (c < cend) {
                    const int row_end = (seg + 1) * L;
                    const int e = min(cend, row_end);
                    run(c, e);
                    checkpoint(e - seg * L);
                    if (e == row_end && seg + 1 < kG) {                  // next row: fresh state, its own A / D / bias
                        ++seg; d += 1;
                        Araw = settle(__ldg(Ap + d));
                        bl2 = splat2((biasp ? __ldg(biasp + d) : 0.f) * kLog2e); A2 = splat2(Araw); D2 = splat2(settle(Dp ? __ldg(Dp + d) : 0.f));
                        h = 0.f; msum = make_float2(0.f, 0.f);
                        xrow += a.xchunks; xc = 0;
                    }
                    c = e;
                }
            }
            // ---- the window's y leaves with one box store; then the stage computed one step earlier is refilled
            fence_proxy_async();                                         // generic-proxy tile writes -> TMA store
            __syncwarp();
            if (lane == 0) {
                tma_box_s2g(&tm_y, ty, c0, srow0);
                bulk_commit();
                bulk_wait_read<1>();                                     // every store but this one has been read out of shared memory
                issue_load();
            }
            ++nstore;
            stage = stage + 1 == ns ? 0 : stage + 1;
        }
    }
    if (lane == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");   // stores complete before the CTA retires
}

template <typename T, int kG>
cudaError_t launch_fwd_cw_g(const CUtensorMap *tm, const CwFwdArgs &a, int grid, bool out_f32, cudaStream_t stream) {
    void (*kernel)(const CUtensorMap, const CUtensorMap, const CUtensorMap, const CwFwdArgs);
    if (a.softplus) kernel = out_f32 ? &ss_fwd_cw_kernel<T, true, true, kG> : &ss_fwd_cw_kernel<T, true, false, kG>;
    else kernel = out_f32 ? &ss_fwd_cw_kernel<T, false, true, kG> : &ss_fwd_cw_kernel<T, false, false, kG>;
    cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, a.smem_bytes);
    if (e != cudaSuccess) return e;
    kernel<<<grid, 32, a.smem_bytes, stream>>>(tm[0], tm[1], tm[2], a);
    return cudaGetLastError();
}

template <typename T>
cudaError_t launch_fwd_cw(const CUtensorMap *tm, const CwFwdArgs &a, int grid, bool out_f32, cudaStream_t stream) {
    if constexpr (sizeof(T) == 2) {
        if (a.g == 2) return launch_fwd_cw_g<T, 2>(tm, a, grid, out_f32, stream);
        if (a.g == 4) return launch_fwd_cw_g<T, 4>(tm, a, grid, out_f32, stream);
    }
    return a.g == 1 ? launch_fwd_cw_g<T, 1>(tm, a, grid, out_f32, stream) : cudaErrorInvalidValue;
}

}  // namespace mia
