// Backward selective scan, COLUMN-WALK row-serial path (d_state == 1) on the block states the column-walk forward leaves
// (scan_fwd_cw.cuh): one lane per row, phase 2 only (no forward re-walk), the row walked from its end in 16-column groups.
//
// Why another backward (measured, gpurun r2f / r2i; ncu of the resident-row kernel, profiles/): scan_bwd_rows.cuh and
// scan_bwd_win.cuh run at 41-43 % issue utilisation with 10-12 warps per SM -- 168 registers per thread (seven 16-token
// quantities kept from the recompute to the suffix loop) and still ~300 bytes of spills (long-scoreboard stalls), a two-warp
// barrier, ~170 instructions of 8-byte cp.async pieces per window.  Here
//   * a group (16 columns of 32 rows) of u, delta and dout is one TMA box each, through a 4-stage ring: lane 0 issues three
//     box loads per group, three groups ahead; du / ddelta replace u / delta in the stage and leave with two box stores; a
//     stage is refilled one step after its stores were committed (cp.async.bulk.wait_group.read 1), so nobody waits;
//   * only a, a h_{t-1} and m (softplus) survive the recompute (48 registers instead of 112): the other per-token factors are
//     re-derived in the suffix loop from them and from u / B, which are still in the stage; dC is reduced over the rows right
//     after the recompute and dB after the suffix loop (two 16-value butterflies, 32 shuffles, instead of one of 32 values);
//   * 128 registers, ~13 KB of shared memory per warp: 15-16 resident one-warp CTAs per SM, no barrier.
// Rows of 392 bytes (L = 196 bf16) are walked g = 4 (or 2) to a tensor-map row exactly like the forward, last row first (columns
// [(g - 1) L, g L) from the end), ...; a group that holds a multiple of L is split between the two rows it touches.
// Reductions over rows (dB, dC): the same transposing butterfly as scan_bwd_rows.cuh, one partial per (32 rows, token) in the
// workspace, folded in a fixed order by the finalize kernel -> deterministic.
// Preconditions (host-checked): as scan_fwd_cw.cuh, block states present, dense 16-byte aligned u / delta / dout / du / ddelta.
#pragma once
#include <cuda.h>

#include <type_traits>

#include "scan_bwd_rows.cuh"
#include "scan_fwd_cw.cuh"
#include "scan_fwd_stream.cuh"

namespace mia {

#ifndef MIA_CW_FMA
#define MIA_CW_FMA 0             // 1: h_t by one FFMA (a_t h_{t-1} off the serial chain); measured slower in the 168-register build (tools/ab_cw.py)
#endif

struct CwRegs {
    float2 a[8], hp[8], m[8];      // a_t, a_t h_{t-1}, softplus(delta + bias) log2e of the 16 tokens
};

// Sum each of 16 per-lane values over the 32 lanes through shared memory: every lane writes its 16 values as one row of a
// [32][20] fp32 scratch (80-byte pitch: the four 16-byte stores of 8 lanes fall into 8 different 16-byte slots), then lane l
// adds value l % 16 over the 16 lanes of its half (column reads; the upper half starts 4 rows further so that the two halves
// use disjoint banks), and one shuffle adds the halves.  4 STS.128 + 16 LDS + 16 FADD + 1 SHFL against 16 SHFL + 16 FADD +
// 30 FSEL for a transposing butterfly; fixed summation order.  Returns the warp total of v[l % 16].
__device__ __forceinline__ float reduce16(const float (&v)[16], const int lane, float *red) {
    float4 *row = reinterpret_cast<float4 *>(red + lane * 20);
#pragma unroll
    for (int i = 0; i < 4; ++i) row[i] = make_float4(v[4 * i], v[4 * i + 1], v[4 * i + 2], v[4 * i + 3]);
    __syncwarp();
    const int half = lane >> 4;
    const float *col = red + half * 16 * 20 + (lane & 15);
    float s0 = 0.f, s1 = 0.f;
#pragma unroll
    for (int k = 0; k < 16; k += 2) {
        s0 += col[((k + 4 * half) & 15) * 20];
        s1 += col[((k + 1 + 4 * half) & 15) * 20];
    }
    __syncwarp();                                                        // the scratch is rewritten by the next reduction
    float s = s0 + s1;
    s += __shfl_xor_sync(0xffffffffu, s, 16);
    return s;
}

// One group (or the part of it that belongs to one row): quads [qlo, qhi) of the 16 columns.  tok0: token of the group's
// first column in the current row (negative for the odd row's head); h0: state entering quad qlo.
template <typename T, typename TO, bool kSoftplus, bool kFull>
__device__ __forceinline__ void cw_bwd_block(const int qlo_in, const int qhi_in, const int tok0, const int lane, const float h0, char *tu, char *td,
                                             const char *to, const SwzRow ri, const SwzRow ro, const int wbi, const int wbo, const float *Bf, const float *Cf,
                                             float *red, float *accB, float *accC, const float2 bl2, const float2 A2, const float2 Aln2, const float2 D2, float &G,
                                             float2 &dA2, float2 &dD2, float2 &db2) {
    constexpr int es = (int)sizeof(T), eo = (int)sizeof(TO);
    const int qlo = kFull ? 0 : qlo_in, qhi = kFull ? 4 : qhi_in;
    const float2 kL2E = splat2(kLog2e), kOne = splat2(1.f);
    const int i16 = lane & 15;
    const bool mine = kFull || (i16 >= 4 * qlo && i16 < 4 * qhi);       // this lane's butterfly slot is a token of the block
    CwRegs R;
    float v[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] = 0.f;
    float h = h0;
    // Tile accesses: one quad (4 tokens) at a time, or -- whole blocks of 2-byte types -- two quads = ONE 16-byte access per tile
    // and lane, which is conflict-free on the swizzled tile where the 8-byte accesses are not (Oct, scan_fwd_rows.cuh).
    constexpr bool kOct = kFull && es == 2 && MIA_CW_OCT;
    constexpr int kNQ = kOct ? 2 : 1, kNP = 2 * kNQ, kNS = 4 / kNQ;
    auto ld_in = [&](const char *tile, const int q0, float2(&f)[kNP]) {
        if constexpr (kOct) Oct<T>::ld(tile + ri.at(wbi + 4 * q0 * es), f);
        else Quad<T>::ld(tile + ri.at(wbi + 4 * q0 * es), *reinterpret_cast<float2(*)[2]>(&f[0]));
    };
    auto ld_dy = [&](const int q0, float2(&f)[kNP]) {
        if constexpr (kOct && eo == 2) {
            Oct<TO>::ld(to + ro.at(wbo + 4 * q0 * eo), f);
        } else {
#pragma unroll
            for (int j = 0; j < kNQ; ++j) Quad<TO>::ld(to + ro.at(wbo + 4 * (q0 + j) * eo), *reinterpret_cast<float2(*)[2]>(&f[2 * j]));
        }
    };
    auto ld_bc = [&](const float *src, const int q0, float2(&f)[kNP]) {
#pragma unroll
        for (int j = 0; j < kNQ; ++j) Quad<float>::ld(reinterpret_cast<const char *>(src + 4 * (q0 + j)), *reinterpret_cast<float2(*)[2]>(&f[2 * j]));
    };
    // ---- recompute a, a h_{t-1}, m of the block from the state entering it; dC_t = sum over rows of dy_t h_t on the way
#pragma unroll
    for (int sI = 0; sI < kNS; ++sI) {
        const int q0 = sI * kNQ;
        if (kFull || (q0 >= qlo && q0 < qhi)) {
            float2 dd[kNP], uu[kNP], Bv[kNP], dy[kNP];
            ld_in(td, q0, dd);
            ld_in(tu, q0, uu);
            ld_bc(Bf, q0, Bv);
            ld_dy(q0, dy);
#pragma unroll
            for (int p = 0; p < kNP; ++p) {
                const int k = 2 * q0 + p;
                float2 m = fma2(dd[p], kL2E, bl2);                      // (delta + bias) log2e
                if (kSoftplus) {
                    const float2 e = make_float2(ex2f(fminf(m.x, 120.f)), ex2f(fminf(m.y, 120.f)));
                    const float2 s = add2(e, kOne);
                    m = make_float2(fmaxf(lg2f(s.x), m.x), fmaxf(lg2f(s.y), m.y));   // softplus log2e
                }
                const float2 av = ex2_2(mul2(m, A2));
                const float2 bv = mul2(mul2(m, uu[p]), Bv[p]);
                float2 hp, hh;
                // a_t h_{t-1}, then h_t
#if MIA_CW_FMA
                hp.x = __fmul_rn(av.x, h); h = fmaf(av.x, h, bv.x); hh.x = h;
                hp.y = __fmul_rn(av.y, h); h = fmaf(av.y, h, bv.y); hh.y = h;
#else
                hp.x = av.x * h; h = hp.x + bv.x; hh.x = h;
                hp.y = av.y * h; h = hp.y + bv.y; hh.y = h;
#endif
                R.a[k] = av; R.hp[k] = hp; R.m[k] = m;
                const float2 dCv = mul2(dy[p], hh);
                v[2 * k] = dCv.x; v[2 * k + 1] = dCv.y;
            }
        }
    }
    const float dCt = reduce16(v, lane, red);
    if (mine && lane < 16) accC[tok0 + i16] = dCt;
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] = 0.f;
    // ---- suffix recurrence G_t = a_t (dy_t C_t + G_{t+1}), gradients of the block
#pragma unroll
    for (int sI = kNS - 1; sI >= 0; --sI) {
        const int q0 = sI * kNQ;
        if (kFull || (q0 >= qlo && q0 < qhi)) {
            float2 dy[kNP], Cv[kNP], Bv[kNP], uu[kNP], du[kNP], dd[kNP];
            ld_dy(q0, dy);
            ld_bc(Cf, q0, Cv);
            ld_bc(Bf, q0, Bv);
            ld_in(tu, q0, uu);                                          // u is still in the stage (du is written below)
#pragma unroll
            for (int p = kNP - 1; p >= 0; --p) {
                const int k = 2 * q0 + p;
                const float2 pc = mul2(dy[p], Cv[p]);
                const float2 ap = mul2(R.a[k], pc);
                float2 gg;
                gg.y = pc.y + G; G = fmaf(R.a[k].y, G, ap.y);
                gg.x = pc.x + G; G = fmaf(R.a[k].x, G, ap.x);
                const float2 dBv = mul2(gg, mul2(R.m[k], uu[p]));
                v[2 * k] = dBv.x; v[2 * k + 1] = dBv.y;
                float2 sg = kL2E;                                       // d m / d (delta + bias) = sigmoid log2e = (1 - 2^-m) log2e
                if (kSoftplus) sg = fma2(ex2_2(make_float2(-R.m[k].x, -R.m[k].y)), make_float2(-kLog2e, -kLog2e), kL2E);
                const float2 qv = fma2(R.hp[k], Aln2, mul2(uu[p], Bv[p]));   // ln2 d h_t / d m_t
                du[p] = fma2(gg, mul2(R.m[k], Bv[p]), mul2(dy[p], D2));
                dd[p] = mul2(gg, mul2(qv, sg));
                db2 = add2(db2, dd[p]);
                dA2 = fma2(gg, mul2(R.m[k], R.hp[k]), dA2);
                dD2 = fma2(dy[p], uu[p], dD2);
            }
            if constexpr (kOct) {
                Oct<T>::st(tu + ri.at(wbi + 4 * q0 * es), du);          // du replaces u, ddelta replaces delta
                Oct<T>::st(td + ri.at(wbi + 4 * q0 * es), dd);
            } else {
                Quad<T>::st(tu + ri.at(wbi + 4 * q0 * es), *reinterpret_cast<float2(*)[2]>(&du[0]));
                Quad<T>::st(td + ri.at(wbi + 4 * q0 * es), *reinterpret_cast<float2(*)[2]>(&dd[0]));
            }
        }
    }
    const float dBt = reduce16(v, lane, red);
    if (mine && lane < 16) accB[tok0 + i16] = dBt * kLn2;
}

// kMinBlk = resident one-warp CTAs per SM the register allocation is sized for: 12 -> 168 registers (three warps per scheduler);
// 8 -> ptxas takes 247 and has no spills: same instructions, scheduled with the loads hoisted further.  The planner runs many
// short items with 8 warps per SM anyway (plan_cw_bwd), so that build costs them no residency.
template <typename T, bool kSoftplus, bool kOutF32, int kG, int kMinBlk>
__global__ void __launch_bounds__(32, kMinBlk) ss_bwd_cw_kernel(const __grid_constant__ CUtensorMap tm_u, const __grid_constant__ CUtensorMap tm_d,
                                                           const __grid_constant__ CUtensorMap tm_o, const __grid_constant__ CUtensorMap tm_du,
                                                           const __grid_constant__ CUtensorMap tm_dd, const __grid_constant__ CwBwdArgs a) {
    // The swizzled tiles need 1024-byte alignment.  The dynamic shared memory of a kernel without static shared memory starts at
    // the CTA's shared window, which is allocated in 1 KB units: asserted once instead of re-aligned at run time (the re-alignment
    // cost a register and ~10 instructions per step).
    extern __shared__ __align__(1024) char smem[];
    if ((smem_u32(smem) & 1023u) != 0) __trap();
    constexpr int es = (int)sizeof(T);
    constexpr int eo = kOutF32 ? 4 : es;
    using TO = typename std::conditional<kOutF32, float, T>::type;
    using raw = typename Cvt<T>::raw;
    constexpr int RBi = kCwWin * es, RBo = kCwWin * eo;                  // tile row bytes: 64 or 128
    constexpr int kTileI = 32 * RBi, kTileO = 32 * RBo;
    const int lane = threadIdx.x;
    float *Bw = reinterpret_cast<float *>(smem + a.off_bc32), *Cw = Bw + kCwWin;
    uint64_t *full = reinterpret_cast<uint64_t *>(smem + a.off_bar);
    const int ns = a.ns;
    if (lane == 0) {
        for (int s = 0; s < ns; ++s) mbar_init(full + s, 1);
        fence_mbar_init();
    }
    __syncwarp();
    const int L = a.L, ncols = kG * L, ngrp = a.ngrp, nwin = a.nwin;
    const int rows_per_item = 32 * kG;
    const int items_per_group = a.rows_per_group / rows_per_item;
    const float *Ap = reinterpret_cast<const float *>(a.A);
    const float *Dp = reinterpret_cast<const float *>(a.D);
    const float *biasp = reinterpret_cast<const float *>(a.delta_bias);
    const SwzRow ri = swz_row<RBi>(lane), ro = swz_row<RBo>(lane);

    auto item_rows = [&](int item, int &b, int &gq, int &row0) {
        const int bt = item % items_per_group;
        const int bg = item / items_per_group;
        gq = bg % a.G; b = bg / a.G;
        row0 = gq * a.rows_per_group + bt * rows_per_item;
    };

    // ---- load stream: (item, window) pairs in the order this CTA computes them (windows from the last one down), ns - 1 ahead
    int ld_item = blockIdx.x, ld_w = nwin - 1, ld_srow0 = 0, ld_stage = 0;
    if (ld_item < a.n_items) { int b, gq, r0; item_rows(ld_item, b, gq, r0); ld_srow0 = (b * a.dim + r0) / kG; }
    auto issue_load = [&]() {                                           // lane 0 only; no-op past the last item
        if (ld_item < a.n_items) {
            char *st = smem + ld_stage * a.stage_bytes;
            mbar_arrive_expect_tx(full + ld_stage, 2u * kTileI + kTileO);
            tma_box_g2s(st, &tm_u, ld_w * kCwWin, ld_srow0, full + ld_stage);
            tma_box_g2s(st + kTileI, &tm_d, ld_w * kCwWin, ld_srow0, full + ld_stage);
            tma_box_g2s(st + 2 * kTileI, &tm_o, ld_w * kCwWin, ld_srow0, full + ld_stage);
            if (--ld_w < 0) {
                ld_w = nwin - 1;
                ld_item += gridDim.x;
                if (ld_item < a.n_items) { int b, gq, r0; item_rows(ld_item, b, gq, r0); ld_srow0 = (b * a.dim + r0) / kG; }
            }
        }
        ld_stage = ld_stage + 1 == ns ? 0 : ld_stage + 1;
    };
    if (lane == 0)
        for (int s = 0; s < ns - 1; ++s) issue_load();

    uint32_t phbits = 0;
    int stage = 0;
    // B / C elements and the two block states of the window about to be computed: prefetched one step ahead by 4-byte cp.async
    // into a two-slot ring in shared memory (NOT into registers: a register live across a block gets spilled, and the spill
    // store waits for the load -- measured: the dominant stall of the first version).
    // Slot: [raw B 128 B][raw C 128 B][block states of the lower group 128 B][of the upper group 128 B].
    constexpr int kEpw = 4 / es, kNw = kCwWin / kEpw;                    // elements per 4-byte word; words per 32 columns (16 or 32)
    char *pf = smem + a.off_pf;
    float *red = reinterpret_cast<float *>(smem + a.off_red);
    const raw *gB = nullptr, *gC = nullptr;                              // B / C rows of the item the prefetch is in
    const float *gh = nullptr;
    auto bc_rows = [&](int item) {
        if (item < a.n_items) {
            int b, gq, r0;
            item_rows(item, b, gq, r0);
            gB = reinterpret_cast<const raw *>(a.B) + (size_t)b * a.B_bs + (size_t)gq * a.B_gs;
            gC = reinterpret_cast<const raw *>(a.C) + (size_t)b * a.C_bs + (size_t)gq * a.C_gs;
            gh = a.hblk + (size_t)item * ngrp * 32 + lane;
        } else {
            gB = nullptr;
        }
    };
    auto cp4 = [&](char *dst, const void *src, bool ok) {                // 4 bytes, zero-filled when !ok
        asm volatile("cp.async.ca.shared.global [%0], [%1], 4, %2;" ::"r"(smem_u32(dst)), "l"(ok ? src : (const void *)a.hblk), "r"(ok ? 4u : 0u)
                     : "memory");
    };
    int pslot = 0;
    auto prefetch = [&](int w) {                                         // into slot `pslot`
        char *sl = pf + pslot * 512;
        const bool live = gB != nullptr;
#pragma unroll
        for (int part = 0; part < 2; ++part) {                           // part 0: B, part 1: C
            // 2-byte types: 16 words per tensor -> lanes 0-15 copy B, lanes 16-31 copy C (one pass); fp32: 32 words each
            const int wd = kNw == 16 ? (lane & 15) : lane;
            const bool mine = kNw == 32 || (lane >> 4) == part;
            if (mine) {
                const int c = w * kCwWin + wd * kEpw;
                int tk = c;                                              // token of column c: c mod L (pairs never straddle a row end: L is even)
#pragma unroll
                for (int i = 1; i < kG; ++i) tk -= tk >= L ? L : 0;
                cp4(sl + part * 128 + wd * 4, (part == 0 ? gB : gC) + tk, live && c < ncols);
            }
        }
        const int j0 = 2 * w;
        cp4(sl + 256 + lane * 4, gh + j0 * 32, live && j0 > 0);
        cp4(sl + 384 + lane * 4, gh + (j0 + 1) * 32, live && j0 + 1 < ngrp);
        cp_async_commit();
    };
    bc_rows(blockIdx.x);
    prefetch(nwin - 1);

    for (int item = blockIdx.x; item < a.n_items; item += gridDim.x) {
        int b, gq, row0;
        item_rows(item, b, gq, row0);
        const int srow0 = (b * a.dim + row0) / kG;
        int seg = kG - 1;                                                // the last row of the tensor-map row first
        int d = row0 + kG * lane + seg;
        float Araw = __ldg(Ap + d);
        float2 bl2 = splat2((biasp ? __ldg(biasp + d) : 0.f) * kLog2e), A2 = splat2(Araw), Aln2 = splat2(Araw * kLn2),
               D2 = splat2(Dp ? __ldg(Dp + d) : 0.f);
        float2 dA2 = make_float2(0.f, 0.f), dD2 = dA2, db2 = dA2;
        float G = 0.f;
        float *accB = a.acc_dB + ((size_t)item * kG + seg) * L, *accC = a.acc_dC + ((size_t)item * kG + seg) * L;
        auto flush_row = [&]() {
            a.part_dA[(size_t)b * a.dim + d] = (dA2.x + dA2.y) * kLn2;
            a.part_dD[(size_t)b * a.dim + d] = dD2.x + dD2.y;
            a.part_dbias[(size_t)b * a.dim + d] = db2.x + db2.y;
        };

        for (int w = nwin - 1; w >= 0; --w) {
            const int c0 = w * kCwWin;
            // B' = B ln2 and C of this window's 32 columns as fp32 (zero past the end); the two block states
            cp_async_wait<0>();
            __syncwarp();
            float hs0, hs1;
            {
                const char *sl = pf + pslot * 512;
                Bw[lane] = Cvt<T>::to_f(*reinterpret_cast<const raw *>(sl + lane * es)) * kLn2;
                Cw[lane] = Cvt<T>::to_f(*reinterpret_cast<const raw *>(sl + 128 + lane * es));
                hs0 = *reinterpret_cast<const float *>(sl + 256 + lane * 4);
                hs1 = *reinterpret_cast<const float *>(sl + 384 + lane * 4);
            }
            pslot ^= 1;
            if (w > 0) {
                prefetch(w - 1);
            } else {
                bc_rows(item + gridDim.x);
                prefetch(nwin - 1);
            }
            __syncwarp();
            mbar_wait(full + stage, (phbits >> stage) & 1u);
            phbits ^= 1u << stage;
            char *tu = smem + stage * a.stage_bytes, *td = tu + kTileI;
            const char *to = tu + 2 * kTileI;
#pragma unroll 1
            for (int half = 1; half >= 0; --half) {                      // the window's two 16-column groups, upper first
                const int cb = c0 + half * kCwGrp;
                if (cb >= ncols) continue;                               // (only the upper group of a row's last window can be empty)
                if (ns == 2 && half == 0 && lane == 0) {
                    // two stages: the stage computed one step ago is the one the NEXT step needs -> refill it half a step early; its
                    // box stores were committed at the end of that step and have had the upper group's block to be read out
                    // (measured, L = 6400, B = 16: 0.85 -> 0.80 ms; with three stages the same early wait costs 7 %: the stores
                    // drain slowly behind the other warps' loads, so there the refill stays at the end of the step)
                    bulk_wait_read<0>();
                    issue_load();
                }
                const float hslot = half ? hs1 : hs0;
                const int wbi = half * kCwGrp * es, wbo = half * kCwGrp * eo;
                const float *Bf = Bw + half * kCwGrp, *Cf = Cw + half * kCwGrp;
                const int hi0 = min(cb + kCwGrp, ncols);                  // columns [cb, hi0) of this group lie inside the tensor-map row
                if (hi0 == cb + kCwGrp && (kG == 1 || cb >= seg * L)) {  // a whole group inside the current row
                    const int tok0 = cb - seg * L;
                    cw_bwd_block<T, TO, kSoftplus, true>(0, 4, tok0, lane, tok0 == 0 ? 0.f : hslot, tu, td, to, ri, ro, wbi, wbo, Bf, Cf, red, accB,
                                                         accC, bl2, A2, Aln2, D2, G, dA2, dD2, db2);
                } else {
                    // partial group (end of the tensor-map row) and / or a group that holds the end of one row and the start of
                    // the next (of several, for rows shorter than a group): sub-blocks from the high columns down, one per row
                    int hi = hi0;
                    while (hi > cb) {
                        const int row_lo = seg * L;                      // first column of the current row
                        if (kG > 1 && hi <= row_lo) {                    // the current row is finished: switch to the one before it
                            flush_row();
                            seg -= 1; d -= 1;                            // fresh suffix state, its own A / D / bias
                            Araw = __ldg(Ap + d);
                            bl2 = splat2((biasp ? __ldg(biasp + d) : 0.f) * kLog2e); A2 = splat2(Araw); Aln2 = splat2(Araw * kLn2);
                            D2 = splat2(Dp ? __ldg(Dp + d) : 0.f);
                            dA2 = make_float2(0.f, 0.f); dD2 = dA2; db2 = dA2; G = 0.f;
                            accB -= L; accC -= L;
                            continue;
                        }
                        const int lo = kG > 1 ? max(cb, row_lo) : cb;
                        // the block state of the group is the state entering column cb: valid for the sub-block that starts there,
                        // unless that column is the first token of the row
                        const float h0 = lo == row_lo ? 0.f : hslot;
                        cw_bwd_block<T, TO, kSoftplus, false>((lo - cb) / 4, (hi - cb) / 4, cb - row_lo, lane, h0, tu, td, to, ri, ro, wbi, wbo, Bf, Cf,
                                                              red, accB, accC, bl2, A2, Aln2, D2, G, dA2, dD2, db2);
                        hi = lo;
                    }
                }
            }
            // ---- du / ddelta leave with two box stores
            fence_proxy_async();
            __syncwarp();
            if (lane == 0) {
                tma_box_s2g(&tm_du, tu, c0, srow0);
                tma_box_s2g(&tm_dd, td, c0, srow0);
                bulk_commit();
                if (ns > 2) {                                            // refill the stage computed one step earlier
                    bulk_wait_read<1>();
                    issue_load();
                }
            }
            stage = stage + 1 == ns ? 0 : stage + 1;
        }
        flush_row();
    }
    if (lane == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
}

template <typename T, int kG, int kMinBlk>
cudaError_t launch_bwd_cw_gm(const CUtensorMap *tm, const CwBwdArgs &a, int grid, bool dout_f32, cudaStream_t stream) {
    void (*kernel)(const CUtensorMap, const CUtensorMap, const CUtensorMap, const CUtensorMap, const CUtensorMap, const CwBwdArgs);
    if (a.softplus) kernel = dout_f32 ? &ss_bwd_cw_kernel<T, true, true, kG, kMinBlk> : &ss_bwd_cw_kernel<T, true, false, kG, kMinBlk>;
    else kernel = dout_f32 ? &ss_bwd_cw_kernel<T, false, true, kG, kMinBlk> : &ss_bwd_cw_kernel<T, false, false, kG, kMinBlk>;
    cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, a.smem_bytes);
    if (e != cudaSuccess) return e;
    kernel<<<grid, 32, a.smem_bytes, stream>>>(tm[0], tm[1], tm[2], tm[3], tm[4], a);
    return cudaGetLastError();
}

template <typename T, int kG>
cudaError_t launch_bwd_cw_g(const CUtensorMap *tm, const CwBwdArgs &a, int grid, bool dout_f32, cudaStream_t stream) {
    return a.wide ? launch_bwd_cw_gm<T, kG, 8>(tm, a, grid, dout_f32, stream) : launch_bwd_cw_gm<T, kG, 12>(tm, a, grid, dout_f32, stream);
}

template <typename T>
cudaError_t launch_bwd_cw(const CUtensorMap *tm, const CwBwdArgs &a, int grid, bool dout_f32, cudaStream_t stream) {
    if constexpr (sizeof(T) == 2) {
        if (a.g == 2) return launch_bwd_cw_g<T, 2>(tm, a, grid, dout_f32, stream);
        if (a.g == 4) return launch_bwd_cw_g<T, 4>(tm, a, grid, dout_f32, stream);
    }
    return a.g == 1 ? launch_bwd_cw_g<T, 1>(tm, a, grid, dout_f32, stream) : cudaErrorInvalidValue;
}

}  // namespace mia
