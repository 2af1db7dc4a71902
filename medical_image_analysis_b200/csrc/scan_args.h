// Host-side contract between the planner (scan_api.cu) and the selective-scan kernels: the tiling constants the planner
// sizes its plans with, the argument block of every kernel family (passed by value as a __grid_constant__ parameter, so
// field order and types are the kernels' parameter layout) and the per-dtype launchers, explicitly instantiated in
// scan_{fwd,bwd}_{bf16,f16,f32}.cu.  Host code only: a file that includes just this header instantiates no kernel.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>

namespace mia {

// warp-scan kernels (scan_fwd.cuh / scan_bwd.cuh)
constexpr int kTok = 8;  // tokens per lane per chunk
constexpr int kMaxStages = 8;
constexpr int kGroupStages = 2;
constexpr int kThreads = 512;     // bwd: 15 consumer warps + 1 producer: 4 warps per SM sub-partition, 128 registers each
constexpr int kThreadsFwd = 512;

// d_state 1 row-serial, streaming, chunk-parallel and column-walk kernels
constexpr int kBlk = 16;   // tokens per recompute block (= values per quantity entering the butterfly)
constexpr int kRowsChunk = 256;   // tokens per staged chunk of a long row = checkpoint spacing of x (kTok * 32)
constexpr int kStreamTok = 32;   // tokens per stage
constexpr int kChunkTok = 256;
constexpr int kCwTok = 32;       // columns per window
constexpr int kCwGrp = 16;       // columns per group = tokens per recompute block
constexpr int kCwWin = 32;       // columns per window = per stage of the ring (two groups)

// d_state > 1 row-serial kernels
constexpr int kRowsNWarps = 4;   // max warps per CTA: each owns a 32-row batch, all share the B / C rows of the (batch, group)
constexpr int kRnWarps = 4;      // warps per CTA = time slices of a row
constexpr int kRnBlk = 8;        // tokens per recompute block
constexpr int kRnOct = 8;        // rows per TMA stage (two quads): 8 L es bytes is a multiple of 16 for every L

// Warp-scan kernels (scan_fwd.cuh / scan_bwd.cuh and their fast variants).
struct ScanArgs {
    // problem
    int batch, dim, L, N, G, delta_dim;
    int rows_per_group, delta_ratio;
    int softplus, has_z, out_f32;      // out_f32: dtype of out/out_z (fwd) or dout/out_saved (bwd) is float
    // tiling
    int RT, RS, split, tiles_per_seg, LPR, CH, n_chunks, n_seg, stages, n_consumer_warps;
    // span-merge flags (the rows of a tile are back to back in global memory -> one TMA span)
    int flat_u, flat_delta, flat_z, flat_dout, flat_osaved, flat_B, flat_C;
    // shared-memory layout (bytes)
    int row_pitch, rowo_pitch, bc_pitch;
    int off_u, off_delta, off_z, off_dout, off_osaved, off_h0, stage_bytes;   // inside a row stage
    int goff_B, goff_C, goff_A, goff_D, goff_bias, gstage_bytes;              // inside a group stage
    int off_groups, off_bars, off_carry, off_red, off_bcf, smem_bytes;        // row stages start at 0; off_bcf: fp32 B/C chunk
                                                                              // of the d_state > 1 fast backward (0 = absent)
    // pointers
    const void *u, *delta, *A, *B, *C, *D, *delta_bias, *z;
    void *out, *out_z;
    float *x;
    const void *dout, *out_saved;
    void *du, *ddelta, *dz;
    float *part_dA, *part_dD, *part_dbias;   // (batch, dim, N) / (batch, dim) / (batch, dim) f32 partials
    float *acc_dB, *acc_dC;                  // d_state 1: (parts, N, L) partials ; warp-scan kernels with d_state > 1: (batch, G, N, Lp) red.add accumulators
    float *ddelta_full;                      // (batch, dim, L) f32 when delta_ratio > 1
    int bc_atomic;
    // strides (elements)
    long long u_bs, u_ds, delta_bs, delta_ds, z_bs, z_ds, A_ds, A_ns;
    long long B_bs, B_gs, B_ns, C_bs, C_gs, C_ns;
    long long out_bs, out_ds, outz_bs, outz_ds;
    long long dout_bs, dout_ds, osaved_bs, osaved_ds;
    long long du_bs, du_ds, dd_bs, dd_ds, dz_bs, dz_ds;
};

struct RowsArgs {
    int batch, dim, L, G, rows_per_group;
    int softplus;
    int Lc, n_lchunks, n_items;          // tokens per staged chunk, chunks per row, (batch, group, 32-row batch) items
    int tile_bytes, bc_bytes, off_bc32, stage_bytes, smem_bytes;   // bc_bytes: one raw B (or C) chunk slot incl. alignment
                                                                   // slack; off_bc32: fp32 copies (B ln2, then C), Lc floats each
    int xchunks, xchunk_tokens;          // checkpoint geometry of x (shared with the warp-scan kernels)
    const void *u, *delta, *A, *B, *C, *D, *delta_bias;
    void *out;
    float *x;
    long long B_bs, B_gs, C_bs, C_gs;    // element strides of B / C (sequence stride is 1, d_state == 1)
};

struct RowsNArgs {
    int batch, dim, L, G, rows_per_group, N;
    int softplus;
    int n_units, units_per_group;         // unit = `warps` consecutive 32-row batches of one (batch, group)
    int warps, tiles_per_warp;            // 4 warps x (u, delta) tiles, or 2 warps x (u, delta, z) with the z gate
    int tile_bytes, off_bc, off_bar, smem_bytes;
    const void *u, *delta, *A, *B, *C, *D, *delta_bias, *z;
    void *out, *out_z;                    // out_z = out * silu(z) (mamba_ssm signature), both written when z is given
    float *x;                             // (batch, dim, 1, 2 N): (prod a_n, h_n) at the row end
    long long A_ds, A_ns, B_bs, B_gs, B_ns, C_bs, C_gs, C_ns;
};

struct StreamArgs {
    int batch, dim, L, G, rows_per_group;
    int softplus;
    int n_items, Lp;                      // Lp: length of the fp32 B' / C rows
    int off_bc32, smem_bytes;
    int xchunks;
    const void *u, *delta, *A, *B, *C, *D, *delta_bias;
    void *out;
    float *x;
    long long B_bs, B_gs, C_bs, C_gs;
};

struct ChunkArgs {
    int batch, dim, L, G, rows_per_group;
    int softplus;
    int n_chunks, n_items;                 // items = 32-row batches x chunks
    int tile_bytes, off_bc32, off_bar, smem_bytes;
    const void *u, *delta, *A, *B, *C, *D, *delta_bias;
    void *out;
    float *x;
    long long B_bs, B_gs, C_bs, C_gs;
};

struct CwFwdArgs {
    int batch, dim, L, G, rows_per_group;
    int softplus;
    int g, n_items, nwin, ngrp, ns;         // rows per tensor-map row; items of 32 g rows; windows / 16-column groups per tensor-map row; stages
    int stage_bytes, off_out, off_bc32, off_bar, smem_bytes;
    int xchunks, xchunk_tokens;             // checkpoint geometry of x (xchunk_tokens is a power of two >= 32)
    const void *A, *B, *C, *D, *delta_bias;
    float *x, *hblk;
    long long B_bs, B_gs, C_bs, C_gs;
    int zero;                               // always 0 (the planner zero-fills the block); see `settle` in the kernel
};

struct RowsBwdArgs {
    int batch, dim, L, G, rows_per_group;
    int softplus;
    int n_items, nblk, n_chunks;           // nblk: checkpoint slots per half of a chunk; n_chunks: 256-token chunks per row
    int t0_pct;                            // percent of a chunk's tokens owned by warp 0
    int tile_bytes, tileo_bytes;            // one [32 x L] tile of u / delta, of dout
    int off_delta, off_dout, off_bc32, off_ck, off_xch, off_bar, smem_bytes;
    int Lp;                                 // L rounded up to kBlk (length of the fp32 B' and C rows)
    const void *u, *delta, *A, *B, *C, *D, *delta_bias, *dout;
    const float *x;                         // forward checkpoints (batch, dim, n_chunks, 2), read when n_chunks > 1
    void *du, *ddelta;
    float *part_dA, *part_dD, *part_dbias, *acc_dB, *acc_dC;
    long long B_bs, B_gs, C_bs, C_gs;
};

struct RowsNBwdArgs {
    int batch, dim, L, G, rows_per_group;
    int softplus, has_z;
    int n_oct, oct_per_cta, oct_per_group;   // work = octets of 8 consecutive rows; CTA c owns [c * oct_per_cta, ...)
    int nblk, Lp;                            // 8-token blocks per row, nblk * 8
    int pitch_s, pitch_bc, pitch_acc;        // scratch row pitch (floats), B / C row pitch (elements), accumulator pitch (floats)
    int max_parts;                           // partial slots per (batch, group) in acc_dB / acc_dC
    int raw_bytes;                           // one raw tensor tile of 8 rows (in / out dtype sized separately below)
    int off_raw_u, off_raw_d, off_raw_o, off_raw_z, off_raw_os;   // raw tiles (u, delta, dout, z, out_saved)
    int off_sm, off_su, off_sy, off_b, off_c, off_acc, off_ck, off_ckm, off_x, off_bar, smem_bytes;
    const void *u, *delta, *A, *B, *C, *D, *delta_bias, *dout, *z, *out_saved;
    void *du, *ddelta, *dz;
    float *part_dA, *part_dD, *part_dbias, *acc_dB, *acc_dC;
    long long A_ds, A_ns, B_bs, B_gs, B_ns, C_bs, C_gs, C_ns;
};

struct CwBwdArgs {
    int batch, dim, L, G, rows_per_group;
    int softplus;
    int g, n_items, ngrp, nwin, ns;         // rows per tensor-map row; items of 32 g rows; 16-column groups / 32-column windows per tensor-map row; stages
    int wide;                               // at most 8 resident warps per SM planned: the build with up to 255 registers per thread
    int stage_bytes, off_bc32, off_pf, off_red, off_bar, smem_bytes;
    const void *A, *B, *C, *D, *delta_bias;
    const float *hblk;
    float *part_dA, *part_dD, *part_dbias, *acc_dB, *acc_dC;
    long long B_bs, B_gs, C_bs, C_gs;
};

template <typename T> cudaError_t launch_fwd_any(const ScanArgs &, int, cudaStream_t);
template <typename T> cudaError_t launch_fwd_rows(const RowsArgs &, int, bool, cudaStream_t);
template <typename T> cudaError_t launch_fwd_rowsn(const RowsNArgs &, int, bool, cudaStream_t);
template <typename T> cudaError_t launch_fwd_stream(const StreamArgs &, int, bool, cudaStream_t);
template <typename T> cudaError_t launch_fwd_chunks(const ChunkArgs &, int, bool, cudaStream_t);
template <typename T> cudaError_t launch_fwd_cw(const CUtensorMap *, const CwFwdArgs &, int, bool, cudaStream_t);
template <typename T> cudaError_t launch_bwd_any(const ScanArgs &, int, cudaStream_t);
template <typename T> cudaError_t launch_bwd_rows(const RowsBwdArgs &, int, bool, cudaStream_t);
template <typename T> cudaError_t launch_bwd_rowsn(const RowsNBwdArgs &, int, bool, cudaStream_t);
template <typename T> cudaError_t launch_bwd_cw(const CUtensorMap *, const CwBwdArgs &, int, bool, cudaStream_t);

}  // namespace mia
