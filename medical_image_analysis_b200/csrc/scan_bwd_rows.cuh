// Backward selective scan, ROW-SERIAL path (d_state == 1): one LANE per row, two warps per [32 rows x chunk] tile set.
//
// A warp owns 32 consecutive rows of one (batch, group): lane r walks the tokens of row r serially, so the scan itself
// costs one FMA per token (no shuffle scans, no idle lanes past the row end) and B[t], C[t] are shared-memory
// broadcasts.  The backward needs h_{t-1} while walking the row from its end, without room for a whole row of fp32
// states per lane.  Two-level recompute:
//   phase 1  forward over the row, keeping only the state at every 16-token block boundary (32 x 4 B per block);
//   phase 2  blocks from last to first: recompute the block's 16 (a, h, ...) into registers from its checkpoint, then
//            run the suffix recurrence G_t = a_t (dy_t C_t + G_{t+1}) backwards through it.
// du / ddelta overwrite the u / delta tiles in shared memory and leave with one bulk store each (coalesced although
// every lane produces a different row).  dA, dD, ddelta_bias are plain per-lane sums.  dB[t], dC[t] are sums over the
// ROWS, i.e. over the lanes: the 32 per-lane values of a block (16 dB + 16 dC) go through a 31-exchange transposing
// butterfly that leaves lane i with the warp total of value i; the per-warp partials are folded in fixed order by
// ss_finalize_kernel (bit-reproducible, like the warp-scan path).
//
// Log2-domain algebra as in scan_bwd_fast.cuh: m = softplus(delta + bias) log2e, a = 2^(m A), B' = B ln2.
// A CTA is two warps that split every chunk in time (see ss_bwd_rows_kernel); rows longer than 256 tokens are walked
// chunk by chunk from the end, the entering state coming from the forward's checkpoints x.
// Preconditions (host-checked, otherwise the warp-scan kernels run): d_state == 1, delta per row, no z, L % 4 == 0,
// rows_per_group % 32 == 0, dense 16-byte aligned u / delta / dout / du / ddelta; L > 256 additionally needs 16-byte
// aligned row pieces and is only chosen while every 32-row batch gets a resident CTA.
#pragma once
#include <cstdio>
#include <cstdlib>
#include <type_traits>

#include "scan_fwd_rows.cuh"

namespace mia {

__device__ __forceinline__ float2 ex2_2(float2 v) { return make_float2(ex2f(v.x), ex2f(v.y)); }

// State of one 16-token block of one row, all in registers (indices are compile-time after unrolling).
struct BlkRegs {
    float2 a[8], h[8], e[8], r[8], w[8], f[8], u[8];
};

// Recompute the forward quantities of quad `q` (4 tokens starting at byte offsets pu/pd, fp32 B' at Bq) of a block.
template <typename T, bool kSoftplus>
__device__ __forceinline__ void recompute_quad(BlkRegs &R, int q, const char *pu, const char *pd, const float *Bq, float &h,
                                               const float2 bl2, const float2 A2, const float2 Aln2) {
    const float2 kL2E = splat2(kLog2e), kOne = splat2(1.f), kLN2 = splat2(kLn2);
    float2 dd[2], uu[2], Bv[2];
    Quad<T>::ld(pd, dd);
    Quad<T>::ld(pu, uu);
    Quad<float>::ld(reinterpret_cast<const char *>(Bq), Bv);
#pragma unroll
    for (int p = 0; p < 2; ++p) {
        const int k = 2 * q + p;
        float2 m = fma2(dd[p], kL2E, bl2);                      // (delta + bias) log2e
        float2 sg = kL2E;
        if (kSoftplus) {
            const float2 e = make_float2(ex2f(fminf(m.x, 120.f)), ex2f(fminf(m.y, 120.f)));
            const float2 s = add2(e, kOne);
            const float2 sl = fma2(e, kLN2, kLN2);              // (1 + e) ln2
            sg = mul2(e, make_float2(rcpf(sl.x), rcpf(sl.y)));  // sigmoid log2e
            m = make_float2(fmaxf(lg2f(s.x), m.x), fmaxf(lg2f(s.y), m.y));
        }
        const float2 av = ex2_2(mul2(m, A2));
        const float2 mu = mul2(m, uu[p]);
        const float2 bv = mul2(mu, Bv[p]);
        float2 hp, hh;
        hp.x = av.x * h; h = fmaf(av.x, h, bv.x); hh.x = h;     // a_t h_{t-1}, then h_t
        hp.y = av.y * h; h = fmaf(av.y, h, bv.y); hh.y = h;
        const float2 qv = fma2(hp, Aln2, mul2(uu[p], Bv[p]));   // ln2 d h_t / d dl_t
        R.a[k] = av; R.h[k] = hh; R.e[k] = mu; R.u[k] = uu[p];
        R.r[k] = mul2(qv, sg);
        R.w[k] = mul2(m, hp);
        R.f[k] = mul2(m, Bv[p]);
    }
}

// One 16-token block of one 32-row batch: recompute from the checkpoint, suffix recurrence, stores, dB/dC butterfly.
template <typename T, typename TO, bool kSoftplus, bool kFull>
__device__ __forceinline__ void bwd_block(const int t0, const int nq_in, const int tend, const int lane, const float h0, char *pu, char *pd,
                                          const char *po, const float *Bf, const float *Cf, float *accB, float *accC,
                                          const float2 bl2, const float2 A2, const float2 Aln2, const float2 D2,
                                          float &G, float2 &dA2, float2 &dD2, float2 &db2) {
    constexpr int es = (int)sizeof(T), eo = (int)sizeof(TO);
    const int nq = kFull ? 4 : nq_in;
    BlkRegs R;
    float v[32];                                 // v[i] = dB term of token t0 + i, v[16 + i] = dC term
#pragma unroll
    for (int i = 0; i < 32; ++i) v[i] = 0.f;
    float h = h0;
#pragma unroll
    for (int q = 0; q < 4; ++q)
        if (kFull || q < nq) recompute_quad<T, kSoftplus>(R, q, pu + (t0 + 4 * q) * es, pd + (t0 + 4 * q) * es, Bf + t0 + 4 * q, h, bl2, A2, Aln2);
#pragma unroll
    for (int q = 3; q >= 0; --q) {
        if (kFull || q < nq) {
            const int t = t0 + 4 * q;
            float2 dy[2], Cv[2], du[2], dd[2];
            Quad<TO>::ld(po + t * eo, dy);
            Quad<float>::ld(reinterpret_cast<const char *>(Cf + t), Cv);
#pragma unroll
            for (int p = 1; p >= 0; --p) {
                const int k = 2 * q + p;
                const float2 pc = mul2(dy[p], Cv[p]);
                const float2 ap = mul2(R.a[k], pc);
                float2 gg;
                gg.y = pc.y + G; G = fmaf(R.a[k].y, G, ap.y);
                gg.x = pc.x + G; G = fmaf(R.a[k].x, G, ap.x);
                const float2 dBv = mul2(gg, R.e[k]), dCv = mul2(dy[p], R.h[k]);
                v[2 * k] = dBv.x; v[2 * k + 1] = dBv.y;
                v[16 + 2 * k] = dCv.x; v[17 + 2 * k] = dCv.y;
                du[p] = fma2(gg, R.f[k], mul2(dy[p], D2));
                dd[p] = mul2(gg, R.r[k]);
                db2 = add2(db2, dd[p]);
                dA2 = fma2(gg, R.w[k], dA2);
                dD2 = fma2(dy[p], R.u[k], dD2);
            }
            Quad<T>::st(pu + t * es, du);        // du replaces u, ddelta replaces delta
            Quad<T>::st(pd + t * es, dd);
        }
    }
    // transposing butterfly: after the step with stride s a lane keeps the half of its values whose index has
    // bit s equal to its own lane bit, summed with the partner's copy -> lane i ends with the warp total of v[i]
#pragma unroll
    for (int s = 16; s >= 1; s >>= 1) {
        const bool up = (lane & s) != 0;
#pragma unroll
        for (int i = 0; i < s; ++i) {
            const float send = up ? v[i] : v[i + s];
            const float keep = up ? v[i + s] : v[i];
            v[i] = keep + __shfl_xor_sync(0xffffffffu, send, s);
        }
    }
    const int tt = t0 + (lane & 15);
    if (kFull || tt < tend) {
        if (lane < 16) accB[tt] = v[0] * kLn2; else accC[tt] = v[0];
    }
}

// Phase 1 of one 16-token block: advances the local state h (and, for the second half of the row, the running sum of
// m and Gs = sum_t (prod_{s<=t} a_s) dy_t C_t, the suffix value the half's first token hands to the first half).
template <typename T, typename TO, bool kSoftplus, bool kSecond, bool kFull>
__device__ __forceinline__ void phase1_block(const int t0, const int nq, const char *pu, const char *pd, const char *po, const float *Bf,
                                             const float *Cf, const float2 bl2, const float2 A2, float &h, float2 &msum, float &P, float &Gs) {
    constexpr int es = (int)sizeof(T), eo = (int)sizeof(TO);
    const float2 kL2E = splat2(kLog2e), kOne = splat2(1.f);
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        if (kFull || q < nq) {
            const int t = t0 + 4 * q;
            float2 dd[2], uu[2], Bv[2], dy[2], Cv[2];
            Quad<T>::ld(pd + t * es, dd);
            Quad<T>::ld(pu + t * es, uu);
            Quad<float>::ld(reinterpret_cast<const char *>(Bf + t), Bv);
            if (kSecond) {
                Quad<TO>::ld(po + t * eo, dy);
                Quad<float>::ld(reinterpret_cast<const char *>(Cf + t), Cv);
            }
#pragma unroll
            for (int p = 0; p < 2; ++p) {
                float2 m = fma2(dd[p], kL2E, bl2);
                if (kSoftplus) {
                    const float2 e = make_float2(ex2f(fminf(m.x, 120.f)), ex2f(fminf(m.y, 120.f)));
                    const float2 s = add2(e, kOne);
                    m = make_float2(fmaxf(lg2f(s.x), m.x), fmaxf(lg2f(s.y), m.y));
                }
                const float2 av = ex2_2(mul2(m, A2));
                const float2 bv = mul2(mul2(m, uu[p]), Bv[p]);
                h = fmaf(av.x, h, bv.x);
                h = fmaf(av.y, h, bv.y);
                if (kSecond) {
                    msum = add2(msum, m);
                    const float2 pc = mul2(dy[p], Cv[p]);
                    P *= av.x; Gs = fmaf(P, pc.x, Gs);
                    P *= av.y; Gs = fmaf(P, pc.y, Gs);
                }
            }
        }
    }
}

// Phase 1 over one warp's half of the row (tokens [tb, tb + 16 (nb - 1) + 4 nq_last), nb blocks aligned to tb),
// starting from h_in (second half: 0): leaves the local state (second half: also the sum of m) entering every block in ck / ckm.
template <typename T, typename TO, bool kSoftplus, bool kSecond>
__device__ __forceinline__ void bwd_phase1(const int tb, const int nb, const int nq_last, const char *pu, const char *pd, const char *po,
                                           const float *Bf, const float *Cf, float *ck, float *ckm, const float2 bl2, const float2 A2,
                                           const float h_in, float &h_out, float &Gs_out, float &P_out) {
    float h = h_in, P = 1.f, Gs = 0.f;
    float2 msum = make_float2(0.f, 0.f);
#pragma unroll 1
    for (int j = 0; j < nb - 1; ++j) {
        ck[j * 32] = h;
        if (kSecond) ckm[j * 32] = msum.x + msum.y;
        phase1_block<T, TO, kSoftplus, kSecond, true>(tb + j * kBlk, 4, pu, pd, po, Bf, Cf, bl2, A2, h, msum, P, Gs);
    }
    if (nb > 0) {                                        // the half's last block may be ragged
        ck[(nb - 1) * 32] = h;
        if (kSecond) ckm[(nb - 1) * 32] = msum.x + msum.y;
        phase1_block<T, TO, kSoftplus, kSecond, false>(tb + (nb - 1) * kBlk, nq_last, pu, pd, po, Bf, Cf, bl2, A2, h, msum, P, Gs);
    }
    h_out = h;
    Gs_out = Gs;
    P_out = P;
}

// CTA = 2 warps sharing one [32 rows x L] tile set: warp 0 owns the first half of the blocks, warp 1 the second half
// (twice the resident warps per byte of shared memory; the single-warp version was latency-bound at 5 warps per SM).
template <typename T, bool kSoftplus, bool kOutF32>
__global__ void __launch_bounds__(64, 5) ss_bwd_rows_kernel(const __grid_constant__ RowsBwdArgs a) {
    extern __shared__ __align__(128) char smem[];
    constexpr int es = (int)sizeof(T);
    constexpr int eo = kOutF32 ? 4 : es;
    using TO = typename std::conditional<kOutF32, float, T>::type;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    char *tu = smem, *td = smem + a.off_delta, *to = smem + a.off_dout;
    float *Bf = reinterpret_cast<float *>(smem + a.off_bc32), *Cf = Bf + a.Lp;
    float *ck = reinterpret_cast<float *>(smem + a.off_ck) + (warp * a.nblk) * 32 + lane;   // ck[j * 32]: local state entering
                                                                                            // block j of this warp's half
    float *ckm = reinterpret_cast<float *>(smem + a.off_ck) + 2 * a.nblk * 32 + lane;       // sum of m before block j (2nd half)
    float *xch = reinterpret_cast<float *>(smem + a.off_xch) + lane;     // [0]: h at the end of half 0, [32]: G entering half 0,
                                                                         // [64..160): dA, dD, dbias partials of warp 1,
                                                                         // [160..224): G entering a chunk (by chunk parity)
    uint64_t *full = reinterpret_cast<uint64_t *>(smem + a.off_bar);
    if (threadIdx.x == 0) { mbar_init(full, 1); fence_mbar_init(); }
    __syncthreads();

    // Rows longer than one 256-token chunk are walked chunk by chunk from the last to the first, the state entering a
    // chunk coming from the forward's checkpoints x and the suffix value G being carried from chunk to chunk.  Within
    // a chunk warp 0 owns tokens [0, T0), warp 1 [T0, len); blocks are aligned to the start of each half, so each half
    // ends with its own (possibly ragged) block.  The second half also accumulates Gs in phase 1: it gets ~48 %.
    const int L = a.L, nch = a.n_chunks;
    const int batches_per_group = a.rows_per_group / 32;
    const float *Ap = reinterpret_cast<const float *>(a.A);
    const float *Dp = reinterpret_cast<const float *>(a.D);
    const float *biasp = reinterpret_cast<const float *>(a.delta_bias);
    // bytes between two rows of a tile: the row itself when the whole [32 x L] tile is one flat copy; one chunk + 16 B
    // for per-row pieces (a 512-byte pitch would put all 32 lanes on the same banks)
    const int pitch = nch == 1 ? L * es : kRowsChunk * es + 16, pitcho = nch == 1 ? L * eo : kRowsChunk * eo + 16;
    char *pu = tu + (size_t)lane * pitch;
    char *pd = td + (size_t)lane * pitch;
    const char *po = to + (size_t)lane * pitcho;
    uint32_t phase = 0;

    for (int item = blockIdx.x; item < a.n_items; item += gridDim.x) {
        const int bt = item % batches_per_group;
        const int bg = item / batches_per_group;
        const int g = bg % a.G, b = bg / a.G;
        const int row0 = g * a.rows_per_group + bt * 32;
        const int d = row0 + lane;
        const float Araw = __ldg(Ap + d);
        const float Dv = Dp ? __ldg(Dp + d) : 0.f;
        const float2 bl2 = splat2((biasp ? __ldg(biasp + d) : 0.f) * kLog2e), A2 = splat2(Araw), Aln2 = splat2(Araw * kLn2), D2 = splat2(Dv);
        const float2 *xrow = reinterpret_cast<const float2 *>(a.x) + ((size_t)b * a.dim + d) * nch;
        float2 dA2 = make_float2(0.f, 0.f), dD2 = dA2, db2 = dA2;
        float Gc = 0.f;                                  // warp 0: G at the first token of the chunk processed last

        for (int c = nch - 1; c >= 0; --c) {
            const int l0 = c * kRowsChunk, len = min(kRowsChunk, L - l0);
            const int T0 = (len * a.t0_pct / 100) / 4 * 4;
            const int tb = warp == 0 ? 0 : T0, tn = warp == 0 ? T0 : len - T0, tend = tb + tn;
            const int nb = (tn + kBlk - 1) / kBlk;
            const int nq_last = (tn - (nb - 1) * kBlk) / 4;              // quads of the half's last block
            const size_t goff = ((size_t)b * a.dim + row0) * L + l0;     // first row of the tile
            if (nch == 1) {
                if (threadIdx.x == 0) {
                    bulk_g2s(tu, (const char *)a.u + goff * es, (uint32_t)(32 * L * es), full);
                    bulk_g2s(td, (const char *)a.delta + goff * es, (uint32_t)(32 * L * es), full);
                    bulk_g2s(to, (const char *)a.dout + goff * eo, (uint32_t)(32 * L * eo), full);
                    mbar_arrive_expect_tx(full, (uint32_t)(32 * L * (2 * es + eo)));
                }
            } else if (warp == 0) {                      // one piece per row and tensor, issued by the row's lane
                const size_t gro = goff + (size_t)lane * L;
                bulk_g2s(pu, (const char *)a.u + gro * es, (uint32_t)(len * es), full);
                bulk_g2s(pd, (const char *)a.delta + gro * es, (uint32_t)(len * es), full);
                bulk_g2s(const_cast<char *>(po), (const char *)a.dout + gro * eo, (uint32_t)(len * eo), full);
                __syncwarp();
                if (lane == 0) mbar_arrive_expect_tx(full, (uint32_t)(32 * len * (2 * es + eo)));
            }
            {
                const typename Cvt<T>::raw *gB = reinterpret_cast<const typename Cvt<T>::raw *>(a.B) + (size_t)b * a.B_bs + (size_t)g * a.B_gs + l0;
                const typename Cvt<T>::raw *gC = reinterpret_cast<const typename Cvt<T>::raw *>(a.C) + (size_t)b * a.C_bs + (size_t)g * a.C_gs + l0;
                for (int i = threadIdx.x; i < a.Lp; i += 64) {
                    Bf[i] = i < len ? Cvt<T>::to_f(__ldg(gB + i)) * kLn2 : 0.f;
                    Cf[i] = i < len ? Cvt<T>::to_f(__ldg(gC + i)) : 0.f;
                }
            }
            const float hc = (warp == 0 && c > 0) ? xrow[c - 1].y : 0.f;   // state entering the chunk (forward checkpoint)
            __syncthreads();                             // B', C rows complete
            mbar_wait(full, phase);
            phase ^= 1;

            // ---- phase 1: states at the block boundaries of this warp's half (warp 1: local, from 0); exchange
            float hend, Gs, Pt;
            if (warp == 0) bwd_phase1<T, TO, kSoftplus, false>(tb, nb, nq_last, pu, pd, po, Bf, Cf, ck, ckm, bl2, A2, hc, hend, Gs, Pt);
            else bwd_phase1<T, TO, kSoftplus, true>(tb, nb, nq_last, pu, pd, po, Bf, Cf, ck, ckm, bl2, A2, 0.f, hend, Gs, Pt);
            float *gslot = xch + 160 + (c & 1) * 32;     // G entering this chunk from the next one (written by warp 0)
            if (warp == 0) xch[0] = hend;
            else {
                const float Gin = c == nch - 1 ? 0.f : *gslot;
                xch[32] = fmaf(Pt, Gin, Gs);             // suffix value handed to the last token of the first half
                Gs = Gin;
            }
            __syncthreads();
            const float hA = warp == 0 ? 0.f : xch[0];   // state entering the second half
            float G = warp == 0 ? xch[32] : Gs;          // a_{t+1} g_{t+1}: what the suffix recurrence hands to token t

            // ---- phase 2: this warp's blocks from last to first.  Only the last block of a half may be ragged: uniform
            // guards, cold code; all the others are straight-line 16-token code the compiler can schedule across tokens
            float *accB = a.acc_dB + (size_t)item * L + l0, *accC = a.acc_dC + (size_t)item * L + l0;
            int j = nb - 1;
            if (nb > 0 && nq_last < 4) {
                const float h0 = warp == 0 ? ck[j * 32] : fmaf(ex2f(Araw * ckm[j * 32]), hA, ck[j * 32]);
                bwd_block<T, TO, kSoftplus, false>(tb + j * kBlk, nq_last, tend, lane, h0, pu, pd, po, Bf, Cf, accB, accC, bl2, A2, Aln2, D2, G, dA2, dD2, db2);
                --j;
            }
#pragma unroll 1
            for (; j >= 0; --j) {
                const float h0 = warp == 0 ? ck[j * 32] : fmaf(ex2f(Araw * ckm[j * 32]), hA, ck[j * 32]);
                bwd_block<T, TO, kSoftplus, true>(tb + j * kBlk, 4, tend, lane, h0, pu, pd, po, Bf, Cf, accB, accC, bl2, A2, Aln2, D2, G, dA2, dD2, db2);
            }
            if (warp == 0) {
                if (c > 0) xch[160 + ((c - 1) & 1) * 32] = G;            // for warp 1, one chunk earlier in the row
            } else if (c == 0) {
                xch[64] = dA2.x + dA2.y; xch[96] = dD2.x + dD2.y; xch[128] = db2.x + db2.y;
            }
            fence_proxy_async();                         // du / ddelta tiles: generic-proxy writes -> bulk store
            __syncthreads();
            if (warp == 0) {
                if (c == 0) {
                    a.part_dA[(size_t)b * a.dim + d] = (dA2.x + dA2.y + xch[64]) * kLn2;
                    a.part_dD[(size_t)b * a.dim + d] = dD2.x + dD2.y + xch[96];
                    a.part_dbias[(size_t)b * a.dim + d] = db2.x + db2.y + xch[128];
                }
                if (nch == 1) {
                    if (lane == 0) {
                        bulk_s2g((char *)a.du + goff * es, tu, (uint32_t)(32 * L * es));
                        bulk_s2g((char *)a.ddelta + goff * es, td, (uint32_t)(32 * L * es));
                        bulk_commit();
                        bulk_wait_read<0>();             // the tiles are refilled next: they must have been read out
                    }
                } else {
                    const size_t gro = goff + (size_t)lane * L;
                    bulk_s2g((char *)a.du + gro * es, pu, (uint32_t)(len * es));
                    bulk_s2g((char *)a.ddelta + gro * es, pd, (uint32_t)(len * es));
                    bulk_commit();
                    bulk_wait_read<0>();
                    __syncwarp();
                }
            }
            // no barrier here: warp 1 only touches B' / C rows (free since the barrier above) until the next one; the
            // tiles are refilled by warp 0 after its wait, the xch slots are rewritten after the next barriers
        }
    }
    asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
}

template <typename T>
cudaError_t launch_bwd_rows(const RowsBwdArgs &a, int grid, bool dout_f32, cudaStream_t stream) {
    void (*kernel)(const RowsBwdArgs);
    if (a.softplus) kernel = dout_f32 ? &ss_bwd_rows_kernel<T, true, true> : &ss_bwd_rows_kernel<T, true, false>;
    else kernel = dout_f32 ? &ss_bwd_rows_kernel<T, false, true> : &ss_bwd_rows_kernel<T, false, false>;
    cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, a.smem_bytes);
    if (e != cudaSuccess) return e;
    kernel<<<grid, 64, a.smem_bytes, stream>>>(a);
    return cudaGetLastError();
}

}  // namespace mia
