// Backward selective scan for d_state = 16 (SS2D's default, every ARM / MambaXray mixer), rows that fit one chunk
// (L <= 256), with or without the z gate of the mamba_ssm signature.  DETERMINISTIC: no atomics, no red.global.
//
// The warp-scan backward (scan_bwd_fastn.cuh) spends 369 instructions per (row, state) on two 5-step shuffle scans and
// adds every row's dB / dC into an L2 accumulator with red.global.add (6.4 GB of reduction traffic per launch at the
// metric's shape, 16x the algorithmic bytes: profiles/README.md, round 1).  Here the recurrence is serial in a lane again:
//
//   lane = (row of a QUAD of 4 consecutive rows, PAIR of states)   -> 4 rows x 8 state pairs = 32 lanes
//
//   * the two states of a lane are the two halves of packed f32x2 registers (FFMA2 / FMUL2 / FADD2): h = a h + b,
//     the suffix recurrence G = a (dy C + G) and every per-(token, state) product are one packed instruction;
//   * everything that does not depend on the state (m = softplus(delta + bias) log2e, u, dy [already gated by silu(z)],
//     and the outputs du, ddelta) lives in a small fp32 scratch per quad, written by a cooperative pre-pass from the raw
//     TMA tile and turned into the output dtype by a post-pass: alignment (odd L = 197) and dtype handling never enter
//     the main loops;
//   * sums over STATES (du, ddelta need sum_n) are 3-step transposing butterflies over the 8 lanes of a row: lane `sp`
//     ends up owning token t0 + sp of its row and does the per-token epilogue (D dy, sigmoid, dD, dbias) once;
//   * sums over ROWS (dB, dC) are 2-step transposing butterflies over the 4 rows of the quad, then plain fp32
//     read-modify-writes into a shared-memory accumulator [16 states][2][L] that is private to the token range of the warp:
//     a CTA is 4 warps that split the row IN TIME (warp w owns a contiguous range of 8-token blocks), so no two warps
//     ever touch the same accumulator element.  The CTA walks a contiguous range of row quads; when the (batch, group)
//     changes the accumulator is written out as one partial and ss_finalize_kernel folds the <= 3 partials of a group in
//     index order -> bit-reproducible.
//   * time split: warps 1..3 run phase 1 from h = 0 and accumulate P = prod a and Gs = sum_t (prod_{s<=t} a_s) dy_t C_t of
//     their range; one barrier later every warp composes the true entering state / suffix value from the (P, h, Gs) of
//     the others (associativity of the scan operator, selective_scan_common.h:91-96) and corrects its 8-token block
//     checkpoints with h_true = h_local + 2^(A sum m) h_in.  Phase 2 recomputes a block forward into registers and runs
//     the suffix recurrence backwards through it.
//
// Tokens past the end of the row are staged as m = 0, u = 0, dy = 0: a = 1, b = 0, no contribution to any sum, so all
// blocks are full 8-token blocks.  Log2 domain as in the other fast paths: m = softplus log2e, a = 2^(m A), e = m u ln2.
// Formulas: scan_bwd.cuh header (== bwd_kernel_oflex.cuh:216-259 of the reference).
//
// Preconditions (host-checked in scan_api.cu, otherwise the warp-scan kernels run): d_state == 16, delta per row,
// L <= 256, dense rows (stride == L) with 16-byte aligned tensors, rows_per_group % 8 == 0.
#pragma once
#include <type_traits>

#include "scan_fwd_rows.cuh"

namespace mia {

// ---- 8 consecutive tokens of two state rows (shared memory, element type T) -> 8 float2 packed over the two states
template <typename T> struct PairRow;
template <> struct PairRow<__nv_bfloat16> {
    static __device__ __forceinline__ void ld(const void *r0, const void *r1, float2 (&v)[8]) {
        const uint4 a = *reinterpret_cast<const uint4 *>(r0), b = *reinterpret_cast<const uint4 *>(r1);
        const uint32_t wa[4] = {a.x, a.y, a.z, a.w}, wb[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            v[2 * i] = make_float2(__uint_as_float(wa[i] << 16), __uint_as_float(wb[i] << 16));
            v[2 * i + 1] = make_float2(__uint_as_float(wa[i] & 0xffff0000u), __uint_as_float(wb[i] & 0xffff0000u));
        }
    }
};
template <> struct PairRow<__half> {
    static __device__ __forceinline__ void ld(const void *r0, const void *r1, float2 (&v)[8]) {
        uint4 a = *reinterpret_cast<const uint4 *>(r0), b = *reinterpret_cast<const uint4 *>(r1);
        const __half2 *ha = reinterpret_cast<const __half2 *>(&a), *hb = reinterpret_cast<const __half2 *>(&b);
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const float2 fa = __half22float2(ha[i]), fb = __half22float2(hb[i]);
            v[2 * i] = make_float2(fa.x, fb.x);
            v[2 * i + 1] = make_float2(fa.y, fb.y);
        }
    }
};
template <> struct PairRow<float> {
    static __device__ __forceinline__ void ld(const void *r0, const void *r1, float2 (&v)[8]) {
        const float4 *pa = reinterpret_cast<const float4 *>(r0), *pb = reinterpret_cast<const float4 *>(r1);
        const float4 a0 = pa[0], a1 = pa[1], b0 = pb[0], b1 = pb[1];
        v[0] = make_float2(a0.x, b0.x); v[1] = make_float2(a0.y, b0.y); v[2] = make_float2(a0.z, b0.z); v[3] = make_float2(a0.w, b0.w);
        v[4] = make_float2(a1.x, b1.x); v[5] = make_float2(a1.y, b1.y); v[6] = make_float2(a1.z, b1.z); v[7] = make_float2(a1.w, b1.w);
    }
};

__device__ __forceinline__ void ld8f(const float *p, float (&v)[8]) {
    const float4 a = reinterpret_cast<const float4 *>(p)[0], b = reinterpret_cast<const float4 *>(p)[1];
    v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
}

// One step of a transposing butterfly: V values per lane, partner at lane distance kBit.  A lane whose bit is set keeps
// the upper half of the indices, the other the lower half, each summed with the partner's copy; the kept half is in v[0 .. V/2).
template <int V, int kBit>
__device__ __forceinline__ void xpose_step(float (&v)[16], const int lane) {
    const bool up = (lane & kBit) != 0;
#pragma unroll
    for (int i = 0; i < V / 2; ++i) {
        const float send = up ? v[i] : v[i + V / 2];
        const float keep = up ? v[i + V / 2] : v[i];
        v[i] = keep + __shfl_xor_sync(0xffffffffu, send, kBit);
    }
}

// element (r, t) of a raw tile staged by stage_span: rows back to back, the tile start keeps its global misalignment
template <typename T>
__device__ __forceinline__ float raw_at(const char *tile, const int idx) {
    return Cvt<T>::to_f(reinterpret_cast<const typename Cvt<T>::raw *>(tile)[idx]);
}

template <typename T, typename TO, bool kSoftplus, bool kHasZ>
__global__ void __launch_bounds__(32 * kRnWarps, 3) ss_bwd_rowsn_kernel(const __grid_constant__ RowsNBwdArgs a) {
    constexpr int kN = 16, kW = kRnWarps;
    extern __shared__ __align__(128) char smem[];
    using raw = typename Cvt<T>::raw;
    using rawo = typename Cvt<TO>::raw;
    constexpr int es = (int)sizeof(T), eo = (int)sizeof(TO);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int rq = lane >> 3, sp = lane & 7;            // row of the quad, state pair
    const int n0 = 2 * sp;
    const int L = a.L, Lp = a.Lp, nblk = a.nblk;
    float *sM = reinterpret_cast<float *>(smem + a.off_sm), *sU = reinterpret_cast<float *>(smem + a.off_su),
          *sY = reinterpret_cast<float *>(smem + a.off_sy);
    raw *Bs = reinterpret_cast<raw *>(smem + a.off_b), *Cs = reinterpret_cast<raw *>(smem + a.off_c);
    float *acc = reinterpret_cast<float *>(smem + a.off_acc);          // [tensor 0: dB, 1: dC][kN][pitch_acc]
    float2 *ck = reinterpret_cast<float2 *>(smem + a.off_ck);           // [nblk][32]: local state entering block j
    float *ckm = reinterpret_cast<float *>(smem + a.off_ckm);           // [nblk][4]: sum of m of the warp's range before block j
    float2 *xh = reinterpret_cast<float2 *>(smem + a.off_x);            // [kW][32] local end state of the warp's range
    float2 *xP = xh + kW * 32;                                          // [kW][32] prod a over the range
    float2 *xG = xP + kW * 32;                                          // [kW][32] Gs of the range
    float2 *xA = xG + kW * 32;                                          // [kW][32] dA partial (units of 1/ln2)
    float2 *xR = xA + kW * 32;                                          // [kW][4]  (dD, dbias) partial per row
    uint64_t *full = reinterpret_cast<uint64_t *>(smem + a.off_bar);
    const char *raw_u = smem + a.off_raw_u, *raw_d = smem + a.off_raw_d, *raw_o = smem + a.off_raw_o;
    const char *raw_z = smem + a.off_raw_z, *raw_os = smem + a.off_raw_os;

    if (tid == 0) { mbar_init(full, 1); fence_mbar_init(); }
    // zero the accumulators, the scratch and the B / C rows once (padding columns must read as finite zeros)
    for (int i = tid; i < (a.off_ck - a.off_sm) / 16; i += blockDim.x) reinterpret_cast<uint4 *>(smem + a.off_sm)[i] = make_uint4(0, 0, 0, 0);
    __syncthreads();

    // this warp's blocks: [jlo, jhi); the remainder goes to the FIRST warps (warp 0 has no Gs to accumulate)
    const int jlo = nblk - ((kW - warp) * nblk) / kW, jhi = nblk - ((kW - warp - 1) * nblk) / kW;
    const float *Ap = reinterpret_cast<const float *>(a.A);
    const float *Dp = reinterpret_cast<const float *>(a.D);
    const float *biasp = reinterpret_cast<const float *>(a.delta_bias);

    const int oct_begin = blockIdx.x * a.oct_per_cta;
    const int oct_end = min(a.n_oct, oct_begin + a.oct_per_cta);
    const size_t tile_elems = (size_t)kRnOct * L;

    auto issue_oct = [&](const int oct) {              // thread 0: stage the 8 rows of every tensor of octet `oct`
        const int bg = oct / a.oct_per_group;
        const int row0 = (bg % a.G) * a.rows_per_group + (oct % a.oct_per_group) * kRnOct;
        const size_t goff = ((size_t)(bg / a.G) * a.dim + row0) * L;
        uint32_t tx = 0;
        bulk_g2s(const_cast<char *>(raw_u), (const char *)a.u + goff * es, (uint32_t)(tile_elems * es), full); tx += (uint32_t)(tile_elems * es);
        bulk_g2s(const_cast<char *>(raw_d), (const char *)a.delta + goff * es, (uint32_t)(tile_elems * es), full); tx += (uint32_t)(tile_elems * es);
        bulk_g2s(const_cast<char *>(raw_o), (const char *)a.dout + goff * eo, (uint32_t)(tile_elems * eo), full); tx += (uint32_t)(tile_elems * eo);
        if (kHasZ) {
            bulk_g2s(const_cast<char *>(raw_z), (const char *)a.z + goff * es, (uint32_t)(tile_elems * es), full); tx += (uint32_t)(tile_elems * es);
            bulk_g2s(const_cast<char *>(raw_os), (const char *)a.out_saved + goff * eo, (uint32_t)(tile_elems * eo), full); tx += (uint32_t)(tile_elems * eo);
        }
        mbar_arrive_expect_tx(full, tx);
    };
    if (tid == 0 && oct_begin < oct_end) issue_oct(oct_begin);

    uint32_t phase = 0;
    int bg_loaded = -1;
    int prev_b = 0, prev_row0 = 0;                      // quad whose du / ddelta still sit in the scratch
    bool have_prev = false;

    // flush the dB / dC accumulators of (batch, group) `bg` as this CTA's partial, then zero them
    auto flush_acc = [&](const int bg) {
        const int c_lo = (int)(((long long)bg * a.oct_per_group) / a.oct_per_cta);
        const int slot = (int)blockIdx.x - c_lo;
        float *gB = a.acc_dB + ((size_t)bg * a.max_parts + slot) * kN * L;
        float *gC = a.acc_dC + ((size_t)bg * a.max_parts + slot) * kN * L;
        for (int i = tid; i < kN * L; i += blockDim.x) {
            const int n = i / L, l = i - n * L;
            float *pb = acc + (size_t)n * a.pitch_acc + l, *pc = pb + (size_t)kN * a.pitch_acc;
            gB[i] = *pb;
            gC[i] = *pc;
            *pb = 0.f; *pc = 0.f;
        }
    };

    // post-pass of the previous quad (scratch -> du / ddelta in the output dtype) fused with the pre-pass of the next one
    // (raw tile -> m, u, dy in the scratch; dz straight to global): same (row, token) -> same thread in both
    auto post_pre = [&](const bool do_pre, const int b, const int row0, const int qi) {
        for (int r = 0; r < 4; ++r) {
            const int d = row0 + r;
            float bias_l2 = 0.f;
            if (do_pre) bias_l2 = (biasp ? __ldg(biasp + d) : 0.f) * kLog2e;
            for (int t = tid; t < Lp; t += blockDim.x) {
                float *pm = sM + r * a.pitch_s + t, *pu = sU + r * a.pitch_s + t, *py = sY + r * a.pitch_s + t;
                if (have_prev && t < L) {
                    const size_t o = ((size_t)prev_b * a.dim + prev_row0 + r) * L + t;
                    reinterpret_cast<raw *>(a.du)[o] = Cvt<T>::from_f(*pu);
                    reinterpret_cast<raw *>(a.ddelta)[o] = Cvt<T>::from_f(*py);
                }
                if (!do_pre) continue;
                float m = 0.f, uv = 0.f, dy = 0.f;
                if (t < L) {
                    const int idx = (qi * 4 + r) * L + t;
                    uv = raw_at<T>(raw_u, idx);
                    m = fmaf(raw_at<T>(raw_d, idx), kLog2e, bias_l2);
                    if (kSoftplus) m = fmaxf(lg2f(1.f + ex2f(fminf(m, 120.f))), m);
                    dy = raw_at<TO>(raw_o, idx);
                    if (kHasZ) {
                        // out_z = y silu(z): dy = dout silu(z); dz = dout y sigmoid(z) (1 + z (1 - sigmoid(z)))  (y = saved out)
                        const float zv = raw_at<T>(raw_z, idx), ov = raw_at<TO>(raw_os, idx);
                        const float sz = rcpf(1.f + ex2f(-zv * kLog2e));
                        const float dsz = dy * sz;
                        reinterpret_cast<raw *>(a.dz)[((size_t)b * a.dim + d) * L + t] = Cvt<T>::from_f(dsz * ov * fmaf(zv, 1.f - sz, 1.f));
                        dy = dsz * zv;
                    }
                }
                *pm = m; *pu = uv; *py = dy;
            }
        }
    };

    for (int oct = oct_begin; oct < oct_end; ++oct) {
        const int bg = oct / a.oct_per_group;
        const int g = bg % a.G, b = bg / a.G;
        const int orow0 = g * a.rows_per_group + (oct % a.oct_per_group) * kRnOct;
        mbar_wait(full, phase);
        phase ^= 1;
        for (int qi = 0; qi < 2; ++qi) {
            const int row0 = orow0 + 4 * qi;
            const int d = row0 + rq;
            // ---- (batch, group) changed: write the previous group's partial out, stage the new B / C rows
            if (qi == 0 && bg != bg_loaded) {
                if (bg_loaded >= 0) flush_acc(bg_loaded);
                bg_loaded = bg;
                const raw *gB = reinterpret_cast<const raw *>(a.B) + (size_t)b * a.B_bs + (size_t)g * a.B_gs;
                const raw *gC = reinterpret_cast<const raw *>(a.C) + (size_t)b * a.C_bs + (size_t)g * a.C_gs;
                for (int i = tid; i < kN * L; i += blockDim.x) {
                    const int n = i / L, l = i - n * L;
                    Bs[(size_t)n * a.pitch_bc + l] = __ldg(gB + (size_t)n * a.B_ns + l);
                    Cs[(size_t)n * a.pitch_bc + l] = __ldg(gC + (size_t)n * a.C_ns + l);
                }
            }
            post_pre(true, b, row0, qi);
            prev_b = b; prev_row0 = row0; have_prev = true;
            __syncthreads();                                            // B1: scratch (+ B / C rows) ready
            if (qi == 1 && tid == 0 && oct + 1 < oct_end) issue_oct(oct + 1);   // the raw tiles are free again

            const float2 A2 = make_float2(__ldg(Ap + (size_t)d * a.A_ds + (size_t)n0 * a.A_ns),
                                          __ldg(Ap + (size_t)d * a.A_ds + (size_t)(n0 + 1) * a.A_ns));
            const float *mrow = sM + rq * a.pitch_s, *urow = sU + rq * a.pitch_s, *yrow = sY + rq * a.pitch_s;
            const raw *B0 = Bs + (size_t)n0 * a.pitch_bc, *B1 = B0 + a.pitch_bc;
            const raw *C0 = Cs + (size_t)n0 * a.pitch_bc, *C1 = C0 + a.pitch_bc;

            // ---- phase 1: local states at the block boundaries of this warp's range (from h = 0), P and Gs of the range
            {
                float2 h2 = make_float2(0.f, 0.f), P2 = make_float2(1.f, 1.f), Gs2 = make_float2(0.f, 0.f);
                float msum = 0.f;
#pragma unroll 1
                for (int j = jlo; j < jhi; ++j) {
                    const int t0 = j * kRnBlk;
                    ck[j * 32 + lane] = h2;
                    if (sp == 0) ckm[j * 4 + rq] = msum;
                    float m[8], uu[8], dy[8];
                    float2 Bv[8], Cv[8];
                    ld8f(mrow + t0, m);
                    ld8f(urow + t0, uu);
                    PairRow<T>::ld(B0 + t0, B1 + t0, Bv);
                    if (warp > 0) { ld8f(yrow + t0, dy); PairRow<T>::ld(C0 + t0, C1 + t0, Cv); }
#pragma unroll
                    for (int k = 0; k < 8; ++k) {
                        const float2 arg = mul2(splat2(m[k]), A2);
                        const float2 av = make_float2(ex2f(arg.x), ex2f(arg.y));
                        h2 = fma2(av, h2, mul2(splat2(m[k] * uu[k] * kLn2), Bv[k]));
                        msum += m[k];
                        if (warp > 0) {
                            P2 = mul2(P2, av);
                            Gs2 = fma2(P2, mul2(splat2(dy[k]), Cv[k]), Gs2);
                        }
                    }
                }
                xh[warp * 32 + lane] = h2;
                xP[warp * 32 + lane] = P2;
                xG[warp * 32 + lane] = Gs2;
            }
            __syncthreads();                                            // B2: (P, h, Gs) of every range visible

            // ---- compose: state entering this warp's range, suffix value entering it from the right
            float2 hin = make_float2(0.f, 0.f), G2 = make_float2(0.f, 0.f);
            for (int w = 0; w < warp; ++w) hin = fma2(xP[w * 32 + lane], hin, xh[w * 32 + lane]);   // xP[0] = 1 (unused factor of 0)
            for (int w = kW - 1; w > warp; --w) G2 = fma2(xP[w * 32 + lane], G2, xG[w * 32 + lane]);

            // ---- phase 2: blocks from last to first
            float2 dA2 = make_float2(0.f, 0.f);
            float dDl = 0.f, dbl = 0.f;
            const float Dv = Dp ? __ldg(Dp + d) : 0.f;
            float *accB = acc, *accC = acc + (size_t)kN * a.pitch_acc;
#pragma unroll 1
            for (int j = jhi - 1; j >= jlo; --j) {
                const int t0 = j * kRnBlk;
                float2 h2 = ck[j * 32 + lane];
                if (warp > 0) {
                    const float ms = ckm[j * 4 + rq];
                    h2 = fma2(make_float2(ex2f(A2.x * ms), ex2f(A2.y * ms)), hin, h2);
                }
                float m[8], e[8], dy[8];
                float2 Bv[8], Cv[8], av[8], ah[8];
                float v[16];
                ld8f(mrow + t0, m);
                ld8f(urow + t0, e);
                ld8f(yrow + t0, dy);
#pragma unroll
                for (int k = 0; k < 8; ++k) e[k] *= m[k] * kLn2;                // dl u  (dl = m ln2)
                PairRow<T>::ld(B0 + t0, B1 + t0, Bv);
                // forward recompute of the block; dC = dy h
#pragma unroll
                for (int k = 0; k < 8; ++k) {
                    const float2 arg = mul2(splat2(m[k]), A2);
                    av[k] = make_float2(ex2f(arg.x), ex2f(arg.y));
                    ah[k] = mul2(av[k], h2);                                   // a_t h_{t-1}
                    h2 = fma2(splat2(e[k]), Bv[k], ah[k]);                      // h_t
                    const float2 dc = mul2(splat2(dy[k]), h2);
                    v[2 * k] = dc.x; v[2 * k + 1] = dc.y;
                }
                // sum over the 4 rows of the quad: lane (rq, sp) keeps tokens t0 + 2 rq, + 1 of its two states
                xpose_step<16, 16>(v, lane);
                xpose_step<8, 8>(v, lane);
                {
                    float2 *p0 = reinterpret_cast<float2 *>(accC + (size_t)n0 * a.pitch_acc + t0 + 2 * rq);
                    float2 *p1 = reinterpret_cast<float2 *>(accC + (size_t)(n0 + 1) * a.pitch_acc + t0 + 2 * rq);
                    float2 c0 = *p0, c1 = *p1;
                    c0.x += v[0]; c1.x += v[1]; c0.y += v[2]; c1.y += v[3];
                    *p0 = c0; *p1 = c1;
                }
                PairRow<T>::ld(C0 + t0, C1 + t0, Cv);
                float s[16];                                                    // s[2k] = sum_n g B, s[2k+1] = sum_n g a h A (this lane's two states)
#pragma unroll
                for (int k = 7; k >= 0; --k) {
                    const float2 g2 = fma2(splat2(dy[k]), Cv[k], G2);          // g_t = dy_t C_t + a_{t+1} g_{t+1}
                    G2 = mul2(av[k], g2);
                    const float2 gB = mul2(g2, Bv[k]);
                    const float2 gah = mul2(g2, ah[k]);
                    s[2 * k] = gB.x + gB.y;
                    s[2 * k + 1] = fmaf(gah.x, A2.x, gah.y * A2.y);
                    dA2 = fma2(gah, splat2(m[k]), dA2);
                    const float2 db = mul2(g2, splat2(e[k]));                  // dB = g dl u
                    v[2 * k] = db.x; v[2 * k + 1] = db.y;
                }
                xpose_step<16, 16>(v, lane);
                xpose_step<8, 8>(v, lane);
                {
                    float2 *p0 = reinterpret_cast<float2 *>(accB + (size_t)n0 * a.pitch_acc + t0 + 2 * rq);
                    float2 *p1 = reinterpret_cast<float2 *>(accB + (size_t)(n0 + 1) * a.pitch_acc + t0 + 2 * rq);
                    float2 c0 = *p0, c1 = *p1;
                    c0.x += v[0]; c1.x += v[1]; c0.y += v[2]; c1.y += v[3];
                    *p0 = c0; *p1 = c1;
                }
                // sum over the 8 state pairs of the row: lane sp keeps (sum g B, sum g a h A) of token t0 + sp
                xpose_step<16, 4>(s, lane);
                xpose_step<8, 2>(s, lane);
                xpose_step<4, 1>(s, lane);
                {
                    const int t = t0 + sp;
                    const float mt = mrow[t], ut = urow[t], dyt = yrow[t];
                    float ddl = fmaf(ut, s[0], s[1]);
                    if (kSoftplus) ddl *= 1.f - ex2f(-mt);                     // sigmoid(x) = 1 - exp(-softplus(x)) = 1 - 2^(-m)
                    const float duv = fmaf(dyt, Dv, mt * kLn2 * s[0]);
                    dbl += ddl;
                    dDl = fmaf(dyt, ut, dDl);
                    __syncwarp();                                               // every lane of the row has read u / dy of this block
                    sU[rq * a.pitch_s + t] = duv;
                    sY[rq * a.pitch_s + t] = ddl;
                }
            }
            // row partials of this warp's range
            xA[warp * 32 + lane] = dA2;
            dDl += __shfl_xor_sync(0xffffffffu, dDl, 1); dbl += __shfl_xor_sync(0xffffffffu, dbl, 1);
            dDl += __shfl_xor_sync(0xffffffffu, dDl, 2); dbl += __shfl_xor_sync(0xffffffffu, dbl, 2);
            dDl += __shfl_xor_sync(0xffffffffu, dDl, 4); dbl += __shfl_xor_sync(0xffffffffu, dbl, 4);
            if (sp == 0) xR[warp * 4 + rq] = make_float2(dDl, dbl);
            __syncthreads();                                            // B3: du / ddelta in the scratch, partials visible
            if (warp == 0) {
                float2 sA = xA[lane];
#pragma unroll
                for (int w = 1; w < kW; ++w) sA = add2(sA, xA[w * 32 + lane]);
                *reinterpret_cast<float2 *>(a.part_dA + ((size_t)b * a.dim + d) * kN + n0) = make_float2(sA.x * kLn2, sA.y * kLn2);
                if (sp == 0) {
                    float2 r = xR[rq];
#pragma unroll
                    for (int w = 1; w < kW; ++w) r = add2(r, xR[w * 4 + rq]);
                    a.part_dD[(size_t)b * a.dim + d] = r.x;
                    a.part_dbias[(size_t)b * a.dim + d] = r.y;
                }
            }
        }
    }
    if (have_prev) post_pre(false, 0, 0, 0);            // outputs of the last quad
    if (bg_loaded >= 0) {
        __syncthreads();
        flush_acc(bg_loaded);
    }
}

template <typename T>
cudaError_t launch_bwd_rowsn(const RowsNBwdArgs &a, int grid, bool dout_f32, cudaStream_t stream) {
    void (*kernel)(const RowsNBwdArgs) = nullptr;
    const bool sp = a.softplus != 0, hz = a.has_z != 0;
#define MIA_PICK(SP, HZ)                                                                                                      \
    (dout_f32 && !std::is_same<T, float>::value ? (void (*)(const RowsNBwdArgs)) & ss_bwd_rowsn_kernel<T, float, SP, HZ>      \
                                                : (void (*)(const RowsNBwdArgs)) & ss_bwd_rowsn_kernel<T, T, SP, HZ>)
    if (sp) kernel = hz ? MIA_PICK(true, true) : MIA_PICK(true, false);
    else kernel = hz ? MIA_PICK(false, true) : MIA_PICK(false, false);
#undef MIA_PICK
    cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, a.smem_bytes);
    if (e != cudaSuccess) return e;
    kernel<<<grid, 32 * kRnWarps, a.smem_bytes, stream>>>(a);
    return cudaGetLastError();
}

}  // namespace mia
