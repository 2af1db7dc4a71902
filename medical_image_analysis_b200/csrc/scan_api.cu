// Host side of libmia_scan.so: argument validation (the reference's TORCH_CHECKs,
// selective_scan_oflex.cpp:152-204 / 245-312), the planner that picks a kernel family and its geometry for a call
// (plan_fwd / plan_bwd, also behind mia_ss_describe_plan and mia_ss_fwd_writes_block_states), one launch per direction,
// the finalize kernel that folds the backward's deterministic partials, and the extern "C" surface declared in
// include/mia_selective_scan.h.  The kernels are reached only through the launchers declared in scan_args.h and
// instantiated in the per-dtype scan_{fwd,bwd}_*.cu files: this file compiles none of them.
#include <algorithm>
#include <atomic>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <initializer_list>
#include <type_traits>

#include "../../include/mia_selective_scan.h"
#include "scan_args.h"
#include "scan_common.cuh"
#include "tma_host.h"

namespace {

thread_local char g_err[512] = "";
std::atomic<uint64_t> g_launches{0};

int fail(int code, const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}

#define MIA_CHECK(cond, ...) \
    do { if (!(cond)) return fail(MIA_EINVAL, __VA_ARGS__); } while (0)
#define MIA_CUDA(expr) \
    do { cudaError_t e__ = (expr); if (e__ != cudaSuccess) return fail(MIA_ECUDA, "%s: %s", #expr, cudaGetErrorString(e__)); } while (0)

// Debugging knobs (force a kernel family, move the half split) exist only in -DMIA_DEBUG builds; the release library
// reads no environment variable and has no mode that alters results.
#ifdef MIA_DEBUG
bool dbg_knob(const char *name) { return getenv(name) != nullptr; }
int dbg_int(const char *name, int dflt) { const char *v = getenv(name); return v ? atoi(v) : dflt; }
#define MIA_TRACE(...) do { if (getenv("MIA_TRACE")) { fprintf(stderr, "[mia] " __VA_ARGS__); fputc('\n', stderr); } } while (0)
#else
#define MIA_TRACE(...) do { } while (0)
constexpr bool dbg_knob(const char *) { return false; }
constexpr int dbg_int(const char *, int dflt) { return dflt; }
#endif

int esize(int dt) { return dt == MIA_F32 ? 4 : 2; }
int round_up(int x, int m) { return (x + m - 1) / m * m; }

struct DeviceInfo { int sms = 0; int smem_optin = 0; };
int device_info(DeviceInfo &di) {
    static thread_local int cached_dev = -1;
    static thread_local DeviceInfo cached;
    int dev = 0;
    MIA_CUDA(cudaGetDevice(&dev));
    if (dev != cached_dev) {
        MIA_CUDA(cudaDeviceGetAttribute(&cached.sms, cudaDevAttrMultiProcessorCount, dev));
        MIA_CUDA(cudaDeviceGetAttribute(&cached.smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
        cached_dev = dev;
    }
    di = cached;
    return MIA_OK;
}

int lanes_per_row(int L) {
    if (L > 128) return 32;
    int need = (L + mia::kTok - 1) / mia::kTok, lpr = 4;
    while (lpr < need) lpr <<= 1;
    return lpr;
}

struct WorkspaceLayout {
    size_t part_dA = 0, part_dD = 0, part_dbias = 0, acc_dB = 0, acc_dC = 0, ddelta_full = 0, total = 0;
    size_t acc_bytes = 0;
    bool bc_atomic = false;
};

// Work plan shared by fwd and bwd (the checkpoint geometry must match between them).
struct Plan {
    int LPR, CH, n_chunks, RPP, NW, RT, RS, split, tiles_per_seg, n_seg;
};

void set_split(Plan &pl, const mia_ss_params &p, int split) {
    const int rpg = p.dim / p.n_groups;
    pl.RS = (rpg + split - 1) / split;
    pl.split = (rpg + pl.RS - 1) / pl.RS;
    pl.tiles_per_seg = (pl.RS + pl.RT - 1) / pl.RT;
    pl.n_seg = p.batch * p.n_groups * pl.split;
}

Plan make_plan(const mia_ss_params &p, int sms, bool bwd) {
    Plan pl;
    pl.LPR = lanes_per_row(p.seqlen);
    pl.CH = pl.LPR * mia::kTok;
    pl.n_chunks = (p.seqlen + pl.CH - 1) / pl.CH;
    pl.RPP = 32 / pl.LPR;
    pl.NW = (bwd ? mia::kThreads : mia::kThreadsFwd) / 32 - 1;
    pl.RT = pl.NW * pl.RPP * (bwd ? 4 : 3);   // row passes per warp and row stage (amortises the per-stage bookkeeping)
    const int rpg = p.dim / p.n_groups;
    // Segments: (batch, group, row range).  Aim at >= ~6 segments per SM with the best last-wave balance; a segment
    // keeps its carries in shared memory, so bound rows * d_state.
    const long long bg = (long long)p.batch * p.n_groups;
    int max_split = (rpg + pl.RPP - 1) / pl.RPP;
    int min_split = 1;
    while ((long long)((rpg + min_split - 1) / min_split) * p.dstate > 4096 && min_split < max_split) ++min_split;
    int want = (int)((6LL * sms + bg - 1) / bg);
    if (want < min_split) want = min_split;
    if (want > max_split) want = max_split;
    int best = want;
    double best_eff = -1.0;
    for (int sp = want; sp <= want + 3 && sp <= max_split; ++sp) {
        Plan t = pl;
        set_split(t, p, sp);
        const double waves = (double)t.n_seg / sms;
        const double eff = waves / (double)((t.n_seg + sms - 1) / sms);
        if (eff > best_eff + 1e-9) { best_eff = eff; best = sp; }
    }
    set_split(pl, p, best);
    return pl;
}

// Work split of the deterministic d_state 16 backward (scan_bwd_rowsn.cuh): sizes only, shared by the workspace query and
// the launch.  Returns false when the shape is not one it takes.
struct RowsNSplit { int n_oct, oct_per_cta, oct_per_group, grid, max_parts; };
bool rowsn_bwd_split(const mia_ss_params &p, int sms, int ctas_per_sm, RowsNSplit &sp) {
    const int rpg = p.dim / p.n_groups;
    if (p.dstate != 16 || p.delta_dim != p.dim || p.seqlen > 256 || (rpg % mia::kRnOct)) return false;
    sp.n_oct = (int)((long long)p.batch * p.dim / mia::kRnOct);
    sp.oct_per_group = rpg / mia::kRnOct;
    const int slots = sms * ctas_per_sm;
    sp.oct_per_cta = (sp.n_oct + slots - 1) / slots;
    sp.grid = (sp.n_oct + sp.oct_per_cta - 1) / sp.oct_per_cta;
    sp.max_parts = (sp.oct_per_group + sp.oct_per_cta - 2) / sp.oct_per_cta + 1;   // CTAs a group's octets can straddle
    return true;
}
constexpr int kRowsNCtasPerSm = 3;   // the split (hence the partial layout) is fixed at 3 CTAs per SM: launching fewer
                                     // resident CTAs (z gate, fp32) only queues them

WorkspaceLayout workspace_layout(const mia_ss_params &p, const Plan &pl, int sms) {
    WorkspaceLayout w;
    auto take = [&](size_t nfloat) { size_t off = w.total; w.total += (nfloat * 4 + 255) / 256 * 256; return off; };
    w.bc_atomic = p.dstate > 1;
    w.part_dA = take((size_t)p.batch * p.dim * p.dstate);
    w.part_dD = take((size_t)p.batch * p.dim);
    w.part_dbias = take((size_t)p.batch * p.dim);
    // d_state == 1: one partial row per segment (warp-scan kernels) or per 32-row batch (row-serial kernel); the query
    // cannot know which of the two will run (it depends on strides and alignment), so size for the larger.
    const int rpg = p.dim / p.n_groups;
    const size_t row_items = (p.dstate == 1 && rpg % 32 == 0) ? (size_t)p.batch * p.n_groups * (rpg / 32) : 0;
    const size_t parts = row_items > (size_t)pl.n_seg ? row_items : (size_t)pl.n_seg;
    size_t nacc = w.bc_atomic ? (size_t)p.batch * p.n_groups * p.dstate * ((p.seqlen + 3) & ~3) : parts * p.dstate * p.seqlen;
    RowsNSplit rs;
    if (rowsn_bwd_split(p, sms, kRowsNCtasPerSm, rs)) {   // whichever d_state 16 kernel runs (it depends on strides), its buffer fits
        const size_t need = (size_t)p.batch * p.n_groups * rs.max_parts * p.dstate * p.seqlen;
        if (need > nacc) nacc = need;
    }
    w.acc_dB = take(nacc);
    w.acc_dC = take(nacc);
    w.acc_bytes = nacc * 4;
    if (p.dim != p.delta_dim) w.ddelta_full = take((size_t)p.batch * p.dim * p.seqlen);
    return w;
}

int validate_sizes(const mia_ss_params &p) {
    MIA_CHECK(p.itype == MIA_F32 || p.itype == MIA_F16 || p.itype == MIA_BF16, "u must be float32, float16 or bfloat16");
    MIA_CHECK(p.otype == p.itype || p.otype == MIA_F32, "out/dout dtype must be the input dtype or float32");
    MIA_CHECK(p.batch > 0 && p.dim > 0 && p.seqlen > 0 && p.dstate > 0 && p.n_groups > 0 && p.delta_dim > 0, "empty or negative size");
    MIA_CHECK(p.dim % p.n_groups == 0, "dims should be dividable by n_groups");
    MIA_CHECK(p.dim % p.delta_dim == 0, "dims should be dividable by delta_dim");
    MIA_CHECK(p.dstate <= 256, "selective_scan only supports state dimension <= 256");
    MIA_CHECK((long long)p.batch * p.dim < (1LL << 31) / 2, "batch*dim too large");
    return MIA_OK;
}

int validate_common(const mia_ss_params &p) {
    if (int rc = validate_sizes(p)) return rc;
    MIA_CHECK(p.u && p.delta && p.A && p.B && p.C, "u, delta, A, B, C must not be null");
    MIA_CHECK(p.n_chunks == mia_ss_num_chunks(p.seqlen), "x must have %d chunks for seqlen %d (got %d)", mia_ss_num_chunks(p.seqlen),
              p.seqlen, p.n_chunks);
    return MIA_OK;
}

void fill_common(mia::ScanArgs &a, const mia_ss_params &p, const Plan &pl) {
    memset(&a, 0, sizeof(a));
    a.batch = p.batch; a.dim = p.dim; a.L = p.seqlen; a.N = p.dstate; a.G = p.n_groups; a.delta_dim = p.delta_dim;
    a.rows_per_group = p.dim / p.n_groups;
    a.delta_ratio = p.dim / p.delta_dim;
    a.softplus = p.delta_softplus; a.has_z = p.z != nullptr; a.out_f32 = (p.otype == MIA_F32) && (p.itype != MIA_F32);
    a.RT = pl.RT; a.RS = pl.RS; a.split = pl.split; a.tiles_per_seg = pl.tiles_per_seg; a.LPR = pl.LPR; a.CH = pl.CH;
    a.n_chunks = pl.n_chunks; a.n_seg = pl.n_seg; a.n_consumer_warps = pl.NW;
    a.u = p.u; a.delta = p.delta; a.A = p.A; a.B = p.B; a.C = p.C; a.D = p.D; a.delta_bias = p.delta_bias; a.z = p.z;
    a.x = p.x;
    a.u_bs = p.u_batch_stride; a.u_ds = p.u_d_stride; a.delta_bs = p.delta_batch_stride; a.delta_ds = p.delta_d_stride;
    a.z_bs = p.z_batch_stride; a.z_ds = p.z_d_stride; a.A_ds = p.A_d_stride; a.A_ns = p.A_dstate_stride;
    a.B_bs = p.B_batch_stride; a.B_gs = p.B_group_stride; a.B_ns = p.B_dstate_stride;
    a.C_bs = p.C_batch_stride; a.C_gs = p.C_group_stride; a.C_ns = p.C_dstate_stride;
    const bool whole = pl.n_chunks == 1;
    a.flat_u = whole && p.u_d_stride == p.seqlen;
    a.flat_delta = whole && p.delta_d_stride == p.seqlen;
    a.flat_z = a.has_z && whole && p.z_d_stride == p.seqlen;
    a.flat_B = whole && p.B_dstate_stride == p.seqlen;
    a.flat_C = whole && p.C_dstate_stride == p.seqlen;
}

// Shared-memory carve-up.  Returns false if not even two row stages fit.
bool layout_smem(mia::ScanArgs &a, int es, int eso, bool bwd, int smem_max) {
    const int span = a.CH < a.L ? a.CH : a.L;
    a.row_pitch = round_up(span * es, 16) + 16;
    a.rowo_pitch = round_up(span * eso, 16) + 16;
    a.bc_pitch = a.row_pitch;
    const int slack = a.CH * 4 + 16;   // an 8-token vector read may run past the last row of a region
    int off = 0;
    auto region = [&](int rows, int pitch) { int o = off; off += round_up(rows * pitch + slack, 128); return o; };
    a.off_u = region(a.RT, a.row_pitch);
    a.off_delta = region(a.RT, a.row_pitch);
    if (a.has_z) a.off_z = region(a.RT, a.row_pitch);
    if (bwd) {
        a.off_dout = region(a.RT, a.rowo_pitch);
        if (a.has_z) a.off_osaved = region(a.RT, a.rowo_pitch);
        a.off_h0 = off; off += round_up(a.RT * a.N * 4, 128);
    }
    a.stage_bytes = off;
    off = 0;
    a.goff_B = region(a.N, a.bc_pitch);
    a.goff_C = region(a.N, a.bc_pitch);
    a.goff_A = off; off += round_up(a.RS * a.N * 4, 128);
    a.goff_D = off; off += round_up(a.RS * 4, 128);
    a.goff_bias = off; off += round_up(a.RS * 4, 128);
    a.gstage_bytes = off;
    const int bars = round_up((2 * mia::kMaxStages + 2 * mia::kGroupStages) * 8, 128);
    const int carry = round_up(bwd ? (2 * a.RS * a.N + 2 * a.RS) * 4 : a.RS * a.N * 8, 128);
    const int red = bwd ? a.n_consumer_warps * 256 * 4 : 0;
    const int fixed = mia::kGroupStages * a.gstage_bytes + bars + carry + red;
    int stages = (smem_max - fixed) / a.stage_bytes;
    if (stages > mia::kMaxStages) stages = mia::kMaxStages;
    if (stages < 2) return false;
    a.stages = stages;
    a.off_groups = stages * a.stage_bytes;
    a.off_bars = a.off_groups + mia::kGroupStages * a.gstage_bytes;
    a.off_carry = a.off_bars + bars;
    a.off_red = a.off_carry + carry;
    a.smem_bytes = a.off_red + red;
    return true;
}

// Pick the work plan and carve shared memory; if it does not fit, first cut segments finer (smaller carries and
// parameter blocks), then halve the row tile.
int plan_and_layout(const mia_ss_params &p, const DeviceInfo &di, bool bwd, Plan &pl, mia::ScanArgs &a) {
    pl = make_plan(p, di.sms, bwd);
    const int es = esize(p.itype), eso = esize(p.otype);
    const int rpg = p.dim / p.n_groups;
    for (;;) {
        fill_common(a, p, pl);
        if (bwd) {
            const bool whole = pl.n_chunks == 1;
            a.flat_dout = whole && p.dout_d_stride == p.seqlen;
            a.flat_osaved = a.has_z && whole && p.out_saved_d_stride == p.seqlen;
        }
        if (layout_smem(a, es, eso, bwd, di.smem_optin)) return MIA_OK;
        if (pl.RS > pl.RT) {
            set_split(pl, p, pl.split * 2 < rpg ? pl.split * 2 : rpg);
        } else {
            MIA_CHECK(pl.RT > pl.RPP, "tile does not fit in shared memory (dstate %d, seqlen %d)", p.dstate, p.seqlen);
            pl.RT = pl.RT / 2 < pl.RPP ? pl.RPP : pl.RT / 2;
            set_split(pl, p, pl.split);
        }
    }
}

// ---- Eligibility rules and argument-block pieces shared by the kernel families
// (batch stride, row stride) pairs of (batch, rows, L) tensors: every row L contiguous tokens, rows back to back
bool dense_rows(const mia_ss_params &p, std::initializer_list<std::pair<long long, long long>> tensors) {
    for (const auto &t : tensors)
        if (t.second != p.seqlen || t.first != (long long)p.dim * p.seqlen) return false;
    return true;
}
bool fwd_rows_dense(const mia_ss_params &p) {          // u, delta, out
    return dense_rows(p, {{p.u_batch_stride, p.u_d_stride}, {p.delta_batch_stride, p.delta_d_stride}, {p.out_batch_stride, p.out_d_stride}});
}
bool bwd_rows_dense(const mia_ss_params &p) {          // u, delta, dout, du, ddelta
    return dense_rows(p, {{p.u_batch_stride, p.u_d_stride}, {p.delta_batch_stride, p.delta_d_stride}, {p.dout_batch_stride, p.dout_d_stride},
                          {p.du_batch_stride, p.du_d_stride}, {p.ddelta_batch_stride, p.ddelta_d_stride}});
}
bool aligned16(std::initializer_list<const void *> ptrs) {
    uintptr_t bits = 0;
    for (const void *q : ptrs) bits |= (uintptr_t)q;
    return (bits & 15) == 0;
}
// The d_state 1 kernels read A as one value per row.
bool a_per_row(const mia_ss_params &p) { return p.A_d_stride == 1 || p.dim == 1; }
// Preconditions of every d_state 1 kernel that gives a lane one row: no z gate, delta per row, whole 32-row batches of one
// group, rows of whole 4-token pieces.
bool lane_per_row(const mia_ss_params &p) {
    return p.dstate == 1 && !p.z && p.delta_dim == p.dim && (p.dim / p.n_groups) % 32 == 0 && p.seqlen % 4 == 0;
}

// Fields every row-serial / column-walk argument block has; the rest of the block starts zeroed.
template <typename R>
void init_args(R &r, const mia_ss_params &p) {
    memset(&r, 0, sizeof(r));
    r.batch = p.batch; r.dim = p.dim; r.L = p.seqlen; r.G = p.n_groups; r.rows_per_group = p.dim / p.n_groups;
    r.softplus = p.delta_softplus;
    r.A = p.A; r.B = p.B; r.C = p.C; r.D = p.D; r.delta_bias = p.delta_bias;
    r.B_bs = p.B_batch_stride; r.B_gs = p.B_group_stride; r.C_bs = p.C_batch_stride; r.C_gs = p.C_group_stride;
}

// Resident CTAs per SM for a kernel of `smem` bytes of dynamic shared memory (1 KB reserved per CTA), at most `cap`.
int resident_ctas(int smem, int cap) {
    const int n = (227 * 1024) / (smem + 1024);
    return n > cap ? cap : n;
}

// Geometry of the column-walk kernels (scan_fwd_cw.cuh / scan_bwd_cw.cuh): g rows per tensor-map row.  A pure function of the
// problem's sizes and dtypes (and the SM count) -- it also fixes the LAYOUT of the block states (hblk), which forward and backward must agree on.
// A tensor-map row must be a multiple of 16 bytes (else the map cannot be encoded); it SHOULD be a multiple of 32 (else every
// other row starts mid-sector and every 64-byte box row touches three sectors instead of two: +19 % DRAM reads measured at
// L = 196 bf16 with g = 2).  2-byte types: the smallest g in {1, 2, 4} with g L a multiple of 16 elements, falling back to a
// smaller legal g when rows_per_group is not a multiple of 32 g or when the item count falls between one and two rounds; g > 1
// only for rows of one checkpoint chunk (L <= 256: the kernels write x at row ends only when they walk several rows per
// lane).  fp32 rows (L % 4 == 0) are always legal: g = 1.
bool cw_geometry(const mia_ss_params &p, int sms, int &g) {
    const int es = esize(p.itype), L = p.seqlen;
    if (!lane_per_row(p)) return false;
    const int rpg = p.dim / p.n_groups;
    if (es == 4) { g = 1; return true; }
    const int want = (L % 16 == 0) ? 1 : (L % 8 == 0) ? 2 : 4;
    // Items are 32 g rows: a larger g halves their number, and a problem that fills the resident slots a little more than once
    // pays a whole second round (measured, gpurun r2fin2, B = 64, L = 196, fp32 out: 1536 items on 1332 - 1480 slots, forward
    // 0.079 -> 0.103 ms) -> take the preferred g when its items fit one round or make at least two, else the next smaller
    // legal one.  (~9 resident warps per SM with fp32 outputs / gradients, 12 otherwise; the same estimate for both directions,
    // since forward and backward must pick the same g.)
    const long long slots = (long long)sms * ((esize(p.otype) == 4) ? 9 : 12);
    int fallback = 0;
    for (int c = want; c >= 1; c >>= 1) {
        if (((long long)c * L * es) % 16) break;                 // not a legal tensor-map row any more
        if (c > 1 && L > 256) continue;
        if (rpg % (32 * c)) continue;
        const long long n_items = (long long)p.batch * p.n_groups * (rpg / (32 * c));
        if (n_items <= slots || n_items >= 2 * slots) { g = c; return true; }
        if (!fallback) fallback = c;
    }
    if (fallback) { g = fallback; return true; }
    return false;
}

// ---- One planner per kernel family: eligibility + argument block + grid.  Each returns false when the shape is not one its
// kernel takes (the caller then tries the next family).

// Row-serial forward (scan_fwd_rows.cuh).
bool plan_rows_fwd(const mia_ss_params &p, const DeviceInfo &di, mia::RowsArgs &r, int &grid) {
    const int es = esize(p.itype), L = p.seqlen;
    if (!lane_per_row(p) || dbg_knob("MIA_NO_ROWS_FWD")) return false;
    if (!fwd_rows_dense(p) || !a_per_row(p) || !aligned16({p.u, p.delta, p.out})) return false;
    init_args(r, p);
    const int budget = 13 * 1024;                               // bytes of one [32 x chunk] tile (8 warps per SM at 2-byte dtypes)
    int Lc = L;
    if (32 * L * es > budget) {
        if ((L * es) % 16) return false;                        // per-row pieces must start 16-byte aligned
        Lc = budget / (32 * es) / 8 * 8;
    }
    r.Lc = Lc; r.n_lchunks = (L + Lc - 1) / Lc;
    r.n_items = p.batch * p.n_groups * (r.rows_per_group / 32);
    r.tile_bytes = round_up(32 * Lc * es, 128);
    r.bc_bytes = 0;
    r.off_bc32 = 2 * r.tile_bytes;
    r.stage_bytes = r.off_bc32 + round_up(2 * Lc * 4, 128);
    r.smem_bytes = r.stage_bytes + 128;
    if (r.smem_bytes > di.smem_optin) return false;
    r.xchunks = mia_ss_num_chunks(L); r.xchunk_tokens = mia_ss_chunk_len(L);
    r.u = p.u; r.delta = p.delta; r.out = p.out; r.x = p.x;
    const int per_sm = di.smem_optin / (r.smem_bytes + 1024) > 0 ? resident_ctas(r.smem_bytes, 8) : 1;
    grid = di.sms * (per_sm < 1 ? 1 : per_sm);
    if (grid > r.n_items) grid = r.n_items;
    return true;
}

// Column-walk forward (scan_fwd_cw.cuh): eligibility, argument block, tensor maps (u, delta, out; not encoded when tm is null).
bool plan_cw_fwd(const mia_ss_params &p, const DeviceInfo &di, mia::CwFwdArgs &r, CUtensorMap *tm, int &grid) {
    const int es = esize(p.itype), eo = esize(p.otype), L = p.seqlen;
    int g = 0;
    if (!cw_geometry(p, di.sms, g) || dbg_knob("MIA_NO_CW_FWD")) return false;
    if (!fwd_rows_dense(p) || !a_per_row(p) || !aligned16({p.u, p.delta, p.out})) return false;
    const int rpg = p.dim / p.n_groups;
    const unsigned long long trows = (unsigned long long)p.batch * p.dim / g, tcols = (unsigned long long)g * L;
    if (tcols >= (1ull << 31) || trows >= (1ull << 31)) return false;
    const int n_items = p.batch * p.n_groups * (rpg / (32 * g));
    // few long rows: the chunk-parallel kernel (scan_fwd_chunks.cuh) has more warps to offer than one per 32 rows
    if (n_items < 4 * di.sms && (L + mia::kChunkTok - 1) / mia::kChunkTok >= 2 && !dbg_knob("MIA_FORCE_CW_FWD")) return false;
    init_args(r, p);
    r.zero = 0;                                                  // (the kernel XORs parameter loads with it: scan_fwd_cw.cuh, settle)
    r.g = g; r.n_items = n_items;
    r.nwin = (g * L + mia::kCwTok - 1) / mia::kCwTok;
    r.ngrp = (g * L + 15) / 16;
    const bool of32 = eo == 4 && es != 4;
    const int tile_i = 32 * mia::kCwTok * es, tile_o = 32 * mia::kCwTok * eo;
    r.stage_bytes = 2 * tile_i;
    // stages: 4 unless 3 gives a better-balanced last round (more resident warps)
    int best_ns = 0;
    double best_eff = -1.0;
    for (int ns = 4; ns >= 3; --ns) {
        const int smem = ns * r.stage_bytes + (of32 ? 2 * tile_o : 0) + 2 * mia::kCwTok * 4 + 8 * ns + 16;
        const int per_sm = resident_ctas(smem, 16);
        if (per_sm < 1) continue;
        const long long slots = (long long)di.sms * per_sm;
        const long long rounds = (n_items + slots - 1) / slots;
        const double eff = (double)n_items / (double)(rounds * slots) * (per_sm >= 8 ? 1.0 : per_sm / 8.0);
        if (eff > best_eff + 0.03) { best_eff = eff; best_ns = ns; }
    }
    if (!best_ns) return false;
    r.ns = dbg_int("MIA_CW_STAGES", best_ns);
    r.off_out = r.ns * r.stage_bytes;
    r.off_bc32 = r.off_out + (of32 ? 2 * tile_o : 0);
    r.off_bar = r.off_bc32 + 2 * mia::kCwTok * 4;
    r.smem_bytes = r.off_bar + 8 * r.ns + 16;
    r.xchunks = mia_ss_num_chunks(L); r.xchunk_tokens = mia_ss_chunk_len(L);
    r.x = p.x; r.hblk = p.hblk;
    const void *ptrs[3] = {p.u, p.delta, p.out};
    for (int i = 0; tm && i < 3; ++i) {
        const int e = i == 2 ? eo : es;
        const int trc = mia::tma_make_2d(&tm[i], ptrs[i], trows, tcols, tcols * e, 32, mia::kCwTok, e, mia::kCwTok * e);
        if (trc != 0) { MIA_TRACE("cw fwd: tensor map %d rejected (CUresult %d)", i, trc); return false; }
    }
    int per_sm = resident_ctas(r.smem_bytes, 16);
    per_sm = std::min(per_sm, dbg_int("MIA_CW_MAXPERSM", per_sm));
    if (per_sm < 1) return false;
    const long long slots = (long long)di.sms * per_sm;
    const long long rounds = (n_items + slots - 1) / slots;
    grid = (int)((n_items + rounds - 1) / rounds);              // equal rounds per CTA
    return true;
}

// Chunk-parallel forward for long rows and few 32-row batches (scan_fwd_chunks.cuh).
bool plan_chunks_fwd(const mia_ss_params &p, const DeviceInfo &di, mia::ChunkArgs &r, int &grid) {
    const int es = esize(p.itype), eo = esize(p.otype), L = p.seqlen;
    if (!lane_per_row(p) || dbg_knob("MIA_NO_ROWS_FWD") || dbg_knob("MIA_NO_CHUNKS_FWD")) return false;
    const int nch = (L + mia::kChunkTok - 1) / mia::kChunkTok;
    if (nch < 2 || mia_ss_chunk_len(L) != mia::kChunkTok || ((L * es) % 16) || ((L * eo) % 16)) return false;
    const int n_batches = p.batch * p.n_groups * (p.dim / p.n_groups / 32);
    if (n_batches >= 4 * di.sms) return false;                 // enough rows: the serial row walk fills the machine
    if (!fwd_rows_dense(p) || !a_per_row(p) || !aligned16({p.u, p.delta, p.out})) return false;
    init_args(r, p);
    r.n_chunks = nch;
    r.n_items = n_batches * nch;
    r.tile_bytes = round_up(32 * (mia::kChunkTok * es + 16), 128);
    r.off_bc32 = 2 * r.tile_bytes;
    r.off_bar = r.off_bc32 + 2 * mia::kChunkTok * 4;
    r.smem_bytes = r.off_bar + 128;
    const int per_sm = resident_ctas(r.smem_bytes, 8);
    if (per_sm < 3) return false;
    r.u = p.u; r.delta = p.delta; r.out = p.out; r.x = p.x;
    grid = di.sms * per_sm;
    if (grid > r.n_items) grid = r.n_items;
    return true;
}

// Streaming row-serial forward (scan_fwd_stream.cuh).
bool plan_stream_fwd(const mia_ss_params &p, const DeviceInfo &di, mia::StreamArgs &r, int &grid) {
    const int es = esize(p.itype), eo = esize(p.otype), L = p.seqlen;
    if (!lane_per_row(p) || dbg_knob("MIA_NO_ROWS_FWD") || dbg_knob("MIA_NO_STREAM_FWD")) return false;
    if (!fwd_rows_dense(p) || !a_per_row(p)) return false;
    const uintptr_t piece = 4 * es - 1, pieceo = 4 * eo - 1;    // every row start is a multiple of one 4-token piece
    if ((((uintptr_t)p.u | (uintptr_t)p.delta) & piece) || ((uintptr_t)p.out & pieceo)) return false;
    if (L > 256 && mia_ss_chunk_len(L) != 256) return false;
    init_args(r, p);
    r.n_items = p.batch * p.n_groups * (r.rows_per_group / 32);
    r.Lp = (L + 3) & ~3;
    const int pitch = mia::kStreamTok * es + 4 * es;
    r.off_bc32 = round_up(2 * 2 * 32 * pitch, 128);             // 2 stages x (u, delta)
    r.smem_bytes = r.off_bc32 + round_up(2 * r.Lp * 4, 128);
    if (r.smem_bytes > di.smem_optin) return false;
    r.xchunks = mia_ss_num_chunks(L);
    r.u = p.u; r.delta = p.delta; r.out = p.out; r.x = p.x;
    const int per_sm = resident_ctas(r.smem_bytes, 16);         // 128 registers per thread
    if (per_sm < 4) return false;
    grid = di.sms * per_sm;
    if (grid > r.n_items) grid = r.n_items;
    return true;
}

// Row-serial forward for d_state 8 / 16 (scan_fwd_rowsn.cuh).
bool plan_rowsn_fwd(const mia_ss_params &p, const DeviceInfo &di, mia::RowsNArgs &r, int &grid) {
    const int es = esize(p.itype), L = p.seqlen, N = p.dstate;
    const int rpg = p.dim / p.n_groups;
    if ((N != 16 && N != 8) || p.delta_dim != p.dim || (rpg % 32) || dbg_knob("MIA_NO_ROWS_FWD")) return false;
    if (mia_ss_num_chunks(L) != 1) return false;                // whole rows, one checkpoint
    if (!fwd_rows_dense(p) || !aligned16({p.u, p.delta, p.out})) return false;
    if (p.z && (!dense_rows(p, {{p.z_batch_stride, p.z_d_stride}, {p.out_z_batch_stride, p.out_z_d_stride}}) || !aligned16({p.z, p.out_z})))
        return false;
    if ((32 * L * es) % 16) return false;
    init_args(r, p);
    r.N = N;
    r.warps = p.z ? 2 : mia::kRowsNWarps;
    r.tiles_per_warp = p.z ? 3 : 2;
    const int W = r.warps;
    r.units_per_group = (rpg / 32 + W - 1) / W;
    r.n_units = p.batch * p.n_groups * r.units_per_group;
    r.tile_bytes = round_up(32 * L * es, 128);
    r.off_bc = W * r.tiles_per_warp * r.tile_bytes;
    r.off_bar = r.off_bc + round_up(2 * L * N * es, 128);
    r.smem_bytes = r.off_bar + 128;
    const int per_sm = (int)(233472 / (r.smem_bytes + 1024));
    if (per_sm < 1 || r.smem_bytes > di.smem_optin) return false;
    r.u = p.u; r.delta = p.delta; r.out = p.out; r.x = p.x; r.z = p.z; r.out_z = p.out_z;
    r.A_ds = p.A_d_stride; r.A_ns = p.A_dstate_stride; r.B_ns = p.B_dstate_stride; r.C_ns = p.C_dstate_stride;
    grid = di.sms * (per_sm > 4 ? 4 : per_sm);
    if (grid > r.n_units) grid = r.n_units;
    return true;
}

// Row-serial backward (scan_bwd_rows.cuh).
bool plan_rows_bwd(const mia_ss_params &p, const DeviceInfo &di, mia::RowsBwdArgs &r, int &grid) {
    const int es = esize(p.itype), eo = esize(p.otype), L = p.seqlen;
    if (!lane_per_row(p) || dbg_knob("MIA_NO_ROWS_BWD")) return false;
    const int CH = mia::kRowsChunk;
    const int nch = (L + CH - 1) / CH;
    // long rows: x must hold a checkpoint every 256 tokens, and the per-row pieces of a tile must be 16-byte aligned
    if (nch > 1 && (mia_ss_chunk_len(L) != CH || !p.x || ((L * es) % 16) || ((L * eo) % 16))) return false;
    if (!bwd_rows_dense(p) || !a_per_row(p) || !aligned16({p.u, p.delta, p.dout, p.du, p.ddelta})) return false;
    init_args(r, p);
    r.n_chunks = nch;
    const int span = nch == 1 ? L : CH;                         // tokens of a row resident at a time
    r.t0_pct = dbg_int("MIA_T0_PCT", 52);   // share of a chunk for the half that has no Gs to accumulate
    const int T0 = (span * r.t0_pct / 100) / 4 * 4;
    const int longer = T0 > span - T0 ? T0 : span - T0;
    r.nblk = (longer + mia::kBlk - 1) / mia::kBlk;
    r.Lp = (span + mia::kBlk - 1) / mia::kBlk * mia::kBlk + mia::kBlk;
    r.n_items = p.batch * p.n_groups * (r.rows_per_group / 32);
    r.tile_bytes = round_up(32 * (span * es + (nch > 1 ? 16 : 0)), 128);
    r.tileo_bytes = round_up(32 * (span * eo + (nch > 1 ? 16 : 0)), 128);
    r.off_delta = r.tile_bytes;
    r.off_dout = 2 * r.tile_bytes;
    r.off_bc32 = r.off_dout + r.tileo_bytes;
    r.off_ck = r.off_bc32 + round_up(2 * r.Lp * 4, 128);
    r.off_xch = r.off_ck + 3 * r.nblk * 128;                    // ck of both halves + ckm
    r.off_bar = r.off_xch + 7 * 128;
    r.smem_bytes = r.off_bar + 128;
    const int per_sm = resident_ctas(r.smem_bytes, 5);          // 64 threads x 168 registers: 3 warps per scheduler
    if (per_sm < 3) return false;                               // too few resident warps to hide the dependent chains
    r.u = p.u; r.delta = p.delta; r.dout = p.dout; r.du = p.du; r.ddelta = p.ddelta; r.x = p.x;
    grid = di.sms * per_sm;
    // Long rows: a CTA walks its 32 rows chunk by chunk and each chunk is latency-bound (load -> phase 1 -> exchange ->
    // phase 2 -> store), so this path only wins while every item gets its own resident CTA (measured on B200, L = 6400:
    // 546 vs 734 us at 0.65 items per slot, 1076 vs 1123 us at 1.3, 2017 vs 1769 us at 2.6).
    if (nch > 1 && r.n_items > grid) return false;
    if (grid > r.n_items) grid = r.n_items;
    return true;
}

// Column-walk backward (scan_bwd_cw.cuh) on the forward's block states: eligibility, argument block, tensor maps (u, delta,
// dout, du, ddelta; not encoded when tm is null).
bool plan_cw_bwd(const mia_ss_params &p, const DeviceInfo &di, mia::CwBwdArgs &r, CUtensorMap *tm, int &grid) {
    const int es = esize(p.itype), eo = esize(p.otype), L = p.seqlen;
    int g = 0;
    if (!p.hblk || !cw_geometry(p, di.sms, g) || dbg_knob("MIA_NO_CW_BWD")) return false;
    // Short rows always; rows of more than one 256-token chunk only with enough 32-row items to fill the SMs.  Measured
    // (B200, runs r2i / r2n, L = 6400, bf16): B = 16 (1536 items) 0.86 ms against 1.77 ms for the warp-scan kernel; B = 4 (384
    // items = 2.6 warps per SM): a one-warp-per-item walk took 0.75 ms against 0.55 ms.
    const long long items32 = (long long)p.batch * (p.dim / 32);
    if (!(L <= mia::kRowsChunk || items32 >= 4LL * di.sms || dbg_knob("MIA_FORCE_CW_BWD"))) return false;
    if (!bwd_rows_dense(p) || !a_per_row(p) || !aligned16({p.u, p.delta, p.dout, p.du, p.ddelta})) return false;
    const unsigned long long trows = (unsigned long long)p.batch * p.dim / g, tcols = (unsigned long long)g * L;
    if (tcols >= (1ull << 31) || trows >= (1ull << 31)) return false;
    if ((((uintptr_t)p.B | (uintptr_t)p.C) & 3) || ((p.B_batch_stride | p.B_group_stride | p.C_batch_stride | p.C_group_stride) * es) % 4) return false;
    init_args(r, p);
    r.g = g;
    r.n_items = p.batch * p.n_groups * (r.rows_per_group / (32 * g));
    r.ngrp = (g * L + mia::kCwGrp - 1) / mia::kCwGrp;
    r.nwin = (g * L + mia::kCwWin - 1) / mia::kCwWin;
    const int tile_i = 32 * mia::kCwWin * es, tile_o = 32 * mia::kCwWin * eo;
    r.stage_bytes = 2 * tile_i + tile_o;
    // Many short rows (at least two rounds of items at 8 per SM) want 8 resident warps per SM (see below) and can afford 3
    // stages; otherwise 2 stages with the half-step-early refill, so that 12 warps per SM fit
    const bool many_short = L <= 256 && r.n_items >= 2LL * 8 * di.sms;
    r.ns = dbg_int("MIA_CW_STAGES", many_short ? 3 : 2);
    r.off_bc32 = r.ns * r.stage_bytes;
    r.off_pf = r.off_bc32 + 2 * mia::kCwWin * 4;                // two 512-byte prefetch slots (raw B, raw C, block states of 2 groups)
    r.off_red = r.off_pf + 1024;                                // [32][20] fp32 scratch of the row reductions
    r.off_bar = r.off_red + 32 * 20 * 4;
    r.smem_bytes = r.off_bar + 8 * r.ns + 16;
    r.hblk = p.hblk;
    const void *ptrs[5] = {p.u, p.delta, p.dout, p.du, p.ddelta};
    for (int i = 0; tm && i < 5; ++i) {
        const int e = i == 2 ? eo : es;
        const int trc = mia::tma_make_2d(&tm[i], ptrs[i], trows, tcols, tcols * e, 32, mia::kCwWin, e, mia::kCwWin * e);
        if (trc != 0) { MIA_TRACE("cw bwd: tensor map %d rejected (CUresult %d)", i, trc); return false; }
    }
    int per_sm = resident_ctas(r.smem_bytes, 12);               // 32 threads x 168 registers: 3 warps per scheduler
    // Many short items: 8 resident warps per SM finish an item 1.8x faster than 12 do (measured, gpurun r2s / r2t, bf16,
    // B = 148: L = 196 0.313 against 0.354 ms, L = 200 0.302 / 0.362, L = 100 0.173 / 0.193, L = 104 0.173 / 0.184), so with
    // at least two rounds of short rows the extra rounds cost less than the contention.  Long rows (L = 1024, B = 32: 0.341
    // against 0.291 ms; L = 6400) want every slot.
    if (many_short && per_sm > 8) per_sm = 8;
    per_sm = std::min(per_sm, dbg_int("MIA_CW_MAXPERSM", per_sm));
    if (per_sm < 1) return false;
    // at most 8 resident warps per SM: the build that may use 255 registers (scan_bwd_cw.cuh, kMinBlk); same results
    r.wide = dbg_int("MIA_CW_WIDE", per_sm <= 8 ? 1 : 0);
    if (r.wide && per_sm > 8) per_sm = 8;
    const long long slots = (long long)di.sms * per_sm;
    const long long rounds = (r.n_items + slots - 1) / slots;
    grid = (int)((r.n_items + rounds - 1) / rounds);             // equal rounds per CTA
    return true;
}

// Deterministic d_state 16 backward (scan_bwd_rowsn.cuh).
bool plan_rowsn_bwd(const mia_ss_params &p, const DeviceInfo &di, mia::RowsNBwdArgs &r, int &grid) {
    const int es = esize(p.itype), eo = esize(p.otype), L = p.seqlen;
    RowsNSplit sp;
    if (!rowsn_bwd_split(p, di.sms, kRowsNCtasPerSm, sp) || dbg_knob("MIA_NO_ROWS_BWD")) return false;
    if (!bwd_rows_dense(p) || !aligned16({p.u, p.delta, p.dout})) return false;
    if (p.z && (!dense_rows(p, {{p.z_batch_stride, p.z_d_stride}, {p.out_saved_batch_stride, p.out_saved_d_stride}, {p.dz_batch_stride, p.dz_d_stride}}) ||
                !aligned16({p.z, p.out_saved})))
        return false;
    init_args(r, p);
    r.has_z = p.z != nullptr;
    r.n_oct = sp.n_oct; r.oct_per_cta = sp.oct_per_cta; r.oct_per_group = sp.oct_per_group; r.max_parts = sp.max_parts;
    r.nblk = (L + mia::kRnBlk - 1) / mia::kRnBlk;
    r.Lp = r.nblk * mia::kRnBlk;
    r.pitch_s = r.Lp + 4;
    r.pitch_acc = r.Lp + 4;
    // B / C rows [16 states][pitch]: consecutive state rows 16 bytes apart modulo 128, so that the 8 state pairs of a
    // quarter warp read 8 different 16-byte bank windows
    r.pitch_bc = r.Lp;
    while ((r.pitch_bc * es) % 128 != 16) r.pitch_bc += 16 / es;
    int off = 0;
    auto take = [&](int bytes) { int o = off; off += round_up(bytes, 128); return o; };
    r.off_raw_u = take(mia::kRnOct * L * es);
    r.off_raw_d = take(mia::kRnOct * L * es);
    r.off_raw_o = take(mia::kRnOct * L * eo);
    if (p.z) { r.off_raw_z = take(mia::kRnOct * L * es); r.off_raw_os = take(mia::kRnOct * L * eo); }
    r.off_sm = take(4 * r.pitch_s * 4);
    r.off_su = take(4 * r.pitch_s * 4);
    r.off_sy = take(4 * r.pitch_s * 4);
    r.off_b = take(16 * r.pitch_bc * es);
    r.off_c = take(16 * r.pitch_bc * es);
    r.off_acc = take(2 * 16 * r.pitch_acc * 4);
    r.off_ck = take(r.nblk * 32 * 8);
    r.off_ckm = take(r.nblk * 4 * 4);
    r.off_x = take((4 * mia::kRnWarps * 32 + mia::kRnWarps * 4) * 8);
    r.off_bar = take(8);
    r.smem_bytes = off;
    if (r.smem_bytes > di.smem_optin) return false;
    r.u = p.u; r.delta = p.delta; r.dout = p.dout; r.z = p.z; r.out_saved = p.out_saved; r.du = p.du; r.ddelta = p.ddelta; r.dz = p.dz;
    r.A_ds = p.A_d_stride; r.A_ns = p.A_dstate_stride; r.B_ns = p.B_dstate_stride; r.C_ns = p.C_dstate_stride;
    grid = sp.grid;
    return true;
}

// ---- Selection: one plan per call and direction, shared by the calls, mia_ss_describe_plan and mia_ss_fwd_writes_block_states.
enum Family { kCw, kChunks, kRows, kStream, kRowsN, kWarpScan };
const char *const kFamilyName[] = {"cw", "chunks", "rows", "stream", "rowsn", "warp_scan"};

struct FwdPlan {
    Family family;
    int grid, smem;
    mia::CwFwdArgs cw;
    mia::ChunkArgs chunks;
    mia::RowsArgs rows;
    mia::StreamArgs stream;
    mia::RowsNArgs rowsn;
    mia::ScanArgs ws;
    CUtensorMap tm[3];
    int launches() const { return family == kChunks ? 3 : 1; }   // the chunk-parallel forward is three kernels
};

// The first family, in order of preference, that takes the shape; the warp-scan kernels take every valid one.
// encode = false: the column-walk tensor maps are not encoded (assumed encodable).  When encoding fails the next family runs.
int plan_fwd(const mia_ss_params &p, const DeviceInfo &di, bool encode, FwdPlan &f) {
    if (plan_cw_fwd(p, di, f.cw, encode ? f.tm : nullptr, f.grid)) { f.family = kCw; f.smem = f.cw.smem_bytes; return MIA_OK; }
    if (plan_chunks_fwd(p, di, f.chunks, f.grid)) { f.family = kChunks; f.smem = f.chunks.smem_bytes; return MIA_OK; }
    if (plan_rows_fwd(p, di, f.rows, f.grid)) { f.family = kRows; f.smem = f.rows.smem_bytes; return MIA_OK; }
    if (plan_stream_fwd(p, di, f.stream, f.grid)) { f.family = kStream; f.smem = f.stream.smem_bytes; return MIA_OK; }
    if (plan_rowsn_fwd(p, di, f.rowsn, f.grid)) { f.family = kRowsN; f.smem = f.rowsn.smem_bytes; return MIA_OK; }
    Plan pl;
    mia::ScanArgs &a = f.ws;
    if (int rc = plan_and_layout(p, di, false, pl, a)) return rc;
    a.out = p.out; a.out_z = p.out_z;
    a.out_bs = p.out_batch_stride; a.out_ds = p.out_d_stride; a.outz_bs = p.out_z_batch_stride; a.outz_ds = p.out_z_d_stride;
    f.family = kWarpScan;
    f.grid = a.n_seg < di.sms ? a.n_seg : di.sms;
    f.smem = a.smem_bytes;
    return MIA_OK;
}

struct BwdPlan {
    Family family;
    int grid, smem;
    mia::CwBwdArgs cw;
    mia::RowsNBwdArgs rowsn;
    mia::RowsBwdArgs rows;
    mia::ScanArgs ws;                 // planned for every call: its work split sizes the workspace
    CUtensorMap tm[5];
    WorkspaceLayout w;
    int parts;                        // dB / dC partial slots per (batch, group) that the finalize folds
    bool atomic;                      // dB / dC accumulate with red.add into the zeroed acc_dB / acc_dC (two memsets)
    int launches() const { return 2 + (atomic ? 2 : 0); }
};

template <typename R>
void set_partials(R &r, const mia::ScanArgs &a) {
    r.part_dA = a.part_dA; r.part_dD = a.part_dD; r.part_dbias = a.part_dbias; r.acc_dB = a.acc_dB; r.acc_dC = a.acc_dC;
}

// The deterministic d_state 16 kernel first, then the column-walk kernel on the forward's block states, the row-serial
// kernel, and the warp-scan kernels for every other valid shape.  Checks the workspace like the call.
int plan_bwd(const mia_ss_params &p, const DeviceInfo &di, bool encode, BwdPlan &b) {
    Plan pl;
    mia::ScanArgs &a = b.ws;
    if (int rc = plan_and_layout(p, di, true, pl, a)) return rc;
    a.dout = p.dout; a.out_saved = p.out_saved; a.du = p.du; a.ddelta = p.ddelta; a.dz = p.dz;
    a.dout_bs = p.dout_batch_stride; a.dout_ds = p.dout_d_stride;
    a.osaved_bs = p.out_saved_batch_stride; a.osaved_ds = p.out_saved_d_stride;
    a.du_bs = p.du_batch_stride; a.du_ds = p.du_d_stride; a.dd_bs = p.ddelta_batch_stride; a.dd_ds = p.ddelta_d_stride;
    a.dz_bs = p.dz_batch_stride; a.dz_ds = p.dz_d_stride;
    const WorkspaceLayout &w = b.w = workspace_layout(p, pl, di.sms);
    if (!p.workspace || p.workspace_bytes < w.total)
        return fail(MIA_EWORKSPACE, "workspace too small: need %zu bytes, got %zu", w.total, p.workspace ? p.workspace_bytes : (size_t)0);
    MIA_CHECK(((uintptr_t)p.workspace & 255) == 0, "workspace must be 256-byte aligned");
    char *ws = (char *)p.workspace;
    a.part_dA = (float *)(ws + w.part_dA); a.part_dD = (float *)(ws + w.part_dD); a.part_dbias = (float *)(ws + w.part_dbias);
    a.acc_dB = (float *)(ws + w.acc_dB); a.acc_dC = (float *)(ws + w.acc_dC);
    a.ddelta_full = (float *)(ws + w.ddelta_full);
    if (plan_rowsn_bwd(p, di, b.rowsn, b.grid)) {
        b.family = kRowsN; b.smem = b.rowsn.smem_bytes; b.parts = b.rowsn.max_parts;
    } else if (plan_cw_bwd(p, di, b.cw, encode ? b.tm : nullptr, b.grid)) {
        b.family = kCw; b.smem = b.cw.smem_bytes; b.parts = b.cw.rows_per_group / 32;
    } else if (plan_rows_bwd(p, di, b.rows, b.grid)) {
        b.family = kRows; b.smem = b.rows.smem_bytes; b.parts = b.rows.rows_per_group / 32;
    } else {
        b.family = kWarpScan; b.grid = a.n_seg < di.sms ? a.n_seg : di.sms; b.smem = a.smem_bytes; b.parts = pl.split;
    }
    set_partials(b.cw, a);
    set_partials(b.rowsn, a);
    set_partials(b.rows, a);
    b.atomic = w.bc_atomic && b.family != kRowsN;
    a.bc_atomic = b.atomic;
    return MIA_OK;
}

// The key=value line of mia_ss_describe_plan.
void describe(const FwdPlan &f, char *buf, size_t n) {
    char geo[96] = "";
    if (f.family == kCw) snprintf(geo, sizeof(geo), " g=%d ns=%d", f.cw.g, f.cw.ns);
    if (f.family == kWarpScan) snprintf(geo, sizeof(geo), " LPR=%d split=%d RT=%d stages=%d", f.ws.LPR, f.ws.split, f.ws.RT, f.ws.stages);
    snprintf(buf, n, "kernel=%s grid=%d smem=%d%s launches=%d", kFamilyName[f.family], f.grid, f.smem, geo, f.launches());
}
void describe(const BwdPlan &b, char *buf, size_t n) {
    char geo[96] = "";
    if (b.family == kCw) snprintf(geo, sizeof(geo), " g=%d ns=%d wide=%d", b.cw.g, b.cw.ns, b.cw.wide);
    if (b.family == kWarpScan) snprintf(geo, sizeof(geo), " LPR=%d split=%d RT=%d stages=%d", b.ws.LPR, b.ws.split, b.ws.RT, b.ws.stages);
    snprintf(buf, n, "kernel=%s grid=%d smem=%d%s parts=%d atomic=%d launches=%d", kFamilyName[b.family], b.grid, b.smem, geo, b.parts,
             b.atomic ? 1 : 0, b.launches());
}

int validate_fwd(const mia_ss_params *pp) {
    if (!pp) return fail(MIA_EINVAL, "null params");
    const mia_ss_params &p = *pp;
    if (int rc = validate_common(p)) return rc;
    MIA_CHECK(p.out && p.x, "out and x must not be null");
    MIA_CHECK(!p.z || p.out_z, "out_z is required when z is given");
    return MIA_OK;
}

int validate_bwd(const mia_ss_params *pp) {
    if (!pp) return fail(MIA_EINVAL, "null params");
    const mia_ss_params &p = *pp;
    if (int rc = validate_common(p)) return rc;
    MIA_CHECK(p.dout && p.du && p.ddelta && p.dA && p.dB && p.dC, "dout, du, ddelta, dA, dB, dC must not be null");
    MIA_CHECK(!p.D || p.dD, "dD is required when D is given");
    MIA_CHECK(!p.delta_bias || p.ddelta_bias, "ddelta_bias is required when delta_bias is given");
    MIA_CHECK(!p.z || (p.dz && p.out_saved), "dz and out_saved are required when z is given");
    MIA_CHECK(p.n_chunks == 1 || p.x, "x is required when the sequence spans more than one chunk");
    return MIA_OK;
}

template <typename F>
auto dispatch(int itype, F &&f) {
    switch (itype) {
        case MIA_F32: return f((float *)nullptr);
        case MIA_F16: return f((__half *)nullptr);
        default: return f((__nv_bfloat16 *)nullptr);
    }
}

// ---------------------------------------------------------------------------------------------
// Finalize: fold the backward's partials in a fixed order (deterministic) and cast to the output dtypes.
struct FinArgs {
    int batch, dim, L, N, G, delta_dim, ratio, tiles, bc_atomic, Lp, has_D, has_bias;
    int oct_per_cta, oct_per_group;          // > 0: partials of scan_bwd_rowsn.cuh, group bg has (c_hi - c_lo + 1) <= tiles of them
    const float *part_dA, *part_dD, *part_dbias, *acc_dB, *acc_dC, *ddelta_full;
    float *dA, *dD, *dbias;
    void *dB, *dC, *ddelta;
    long long dA_ds, dA_ns, dB_bs, dB_gs, dB_ns, dC_bs, dC_gs, dC_ns, dd_bs, dd_ds;
    long long n_bc, n_dA, n_dD, n_db, n_dd;
};

// thread items: dB, dC (sum of the per-segment partials / cast of the atomic accumulator) and the ddelta group fold;
// warp items: dA, dD, dbias (sum over the batch, lanes stride over b, shuffle-reduced in a fixed order).
template <typename T>
__global__ void ss_finalize_kernel(const __grid_constant__ FinArgs f) {
    using raw = typename mia::Cvt<T>::raw;
    const long long n_thread_items = 2 * f.n_bc + f.n_dd;
    const long long t1 = (n_thread_items + 31) / 32 * 32;
    const long long n_warp_items = f.n_dA + f.n_dD + f.n_db;
    const long long total = t1 + 32 * n_warp_items;
    for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long long)gridDim.x * blockDim.x) {
        if (idx < t1) {
            long long i = idx;
            if (i >= n_thread_items) continue;
            if (i < 2 * f.n_bc) {
                const bool isC = i >= f.n_bc;
                if (isC) i -= f.n_bc;
                const int l = (int)(i % f.L);
                long long t = i / f.L;
                const int n = (int)(t % f.N); t /= f.N;
                const int g = (int)(t % f.G);
                const int b = (int)(t / f.G);
                const float *acc = isC ? f.acc_dC : f.acc_dB;
                float sum = 0.f;
                if (f.bc_atomic) {
                    sum = acc[((size_t)(b * f.G + g) * f.N + n) * f.Lp + l];
                } else {
                    const float *p0 = acc + (((size_t)(b * f.G + g) * f.tiles) * f.N + n) * f.L + l;
                    const size_t step = (size_t)f.N * f.L;
                    int nt = f.tiles;
                    if (f.oct_per_cta > 0) {             // partial slots actually written for this group (CTAs it straddles)
                        const long long o0 = (long long)(b * f.G + g) * f.oct_per_group;
                        nt = (int)((o0 + f.oct_per_group - 1) / f.oct_per_cta - o0 / f.oct_per_cta) + 1;
                    }
#pragma unroll 4
                    for (int tl = 0; tl < nt; ++tl) sum += p0[tl * step];
                }
                raw *dst = reinterpret_cast<raw *>(isC ? f.dC : f.dB);
                const long long o = isC ? (b * f.dC_bs + g * f.dC_gs + n * f.dC_ns + l) : (b * f.dB_bs + g * f.dB_gs + n * f.dB_ns + l);
                dst[o] = mia::Cvt<T>::from_f(sum);
            } else {   // ddelta fold over the delta group (selective_scan_oflex.cpp:348-350)
                i -= 2 * f.n_bc;
                const int l = (int)(i % f.L);
                long long t = i / f.L;
                const int dg = (int)(t % f.delta_dim);
                const int b = (int)(t / f.delta_dim);
                float sum = 0.f;
                for (int r = 0; r < f.ratio; ++r) sum += f.ddelta_full[((size_t)b * f.dim + dg * f.ratio + r) * f.L + l];
                reinterpret_cast<raw *>(f.ddelta)[b * f.dd_bs + dg * f.dd_ds + l] = mia::Cvt<T>::from_f(sum);
            }
            continue;
        }
        // ---- warp items (idx - t1 is warp aligned, so the whole warp takes this path together)
        long long w = (idx - t1) >> 5;
        const int lane = (int)(idx & 31);
        float sum = 0.f;
        float *dst;
        if (w < f.n_dA) {
            const int n = (int)(w % f.N), d = (int)(w / f.N);
            for (int b = lane; b < f.batch; b += 32) sum += f.part_dA[((size_t)b * f.dim + d) * f.N + n];
            dst = f.dA + d * f.dA_ds + n * f.dA_ns;
        } else if (w < f.n_dA + f.n_dD) {
            w -= f.n_dA;
            for (int b = lane; b < f.batch; b += 32) sum += f.part_dD[(size_t)b * f.dim + w];
            dst = f.dD + w;
        } else {
            w -= f.n_dA + f.n_dD;
            for (int k = lane; k < f.batch * f.ratio; k += 32) {
                const int b = k / f.ratio, r = k - b * f.ratio;
                sum += f.part_dbias[(size_t)b * f.dim + w * f.ratio + r];
            }
            dst = f.dbias + w;
        }
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, off);
        if (lane == 0) *dst = sum;
    }
}

}  // namespace

// =================================================================================================
extern "C" {

int mia_abi_version(void) { return MIA_ABI_VERSION; }
const char *mia_last_error(void) { return g_err; }
uint64_t mia_launch_count(void) { return g_launches.load(); }

int mia_ss_chunk_len(int seqlen) { return lanes_per_row(seqlen) * mia::kTok; }
int mia_ss_num_chunks(int seqlen) {
    const int ch = mia_ss_chunk_len(seqlen);
    return (seqlen + ch - 1) / ch;
}

size_t mia_ss_block_state_floats(const mia_ss_params *pp) {
    if (!pp || validate_sizes(*pp) != MIA_OK) return 0;
    const mia_ss_params &p = *pp;
    if (p.dstate != 1 || ((p.dim / p.n_groups) % 32)) return 0;
    return (size_t)p.batch * p.dim * ((p.seqlen + 15) / 16);
}

int mia_ss_fwd_writes_block_states(const mia_ss_params *pp) {
    if (!pp || !pp->hblk || validate_sizes(*pp) != MIA_OK || !pp->u || !pp->delta || !pp->out) return 0;
    DeviceInfo di;
    if (device_info(di) != MIA_OK) return 0;
    FwdPlan f;                                                   // the maps are encoded: a map the driver rejects means no cw
    return plan_fwd(*pp, di, true, f) == MIA_OK && f.family == kCw ? 1 : 0;   // the column-walk forward is the kernel that fills hblk
}

int mia_ss_describe_plan(const mia_ss_params *pp, int backward, int sms, int smem_optin, char *buf, size_t buf_len) {
    if (int rc = backward ? validate_bwd(pp) : validate_fwd(pp)) return rc;
    MIA_CHECK(buf && buf_len > 0, "no buffer for the plan");
    DeviceInfo di;
    if (sms <= 0 || smem_optin <= 0) {
        if (int rc = device_info(di)) return rc;
    }
    if (sms > 0) di.sms = sms;
    if (smem_optin > 0) di.smem_optin = smem_optin;
    if (backward) {
        BwdPlan b;
        if (int rc = plan_bwd(*pp, di, false, b)) return rc;
        describe(b, buf, buf_len);
    } else {
        FwdPlan f;
        if (int rc = plan_fwd(*pp, di, false, f)) return rc;
        describe(f, buf, buf_len);
    }
    return MIA_OK;
}

int mia_selective_scan_fwd(const mia_ss_params *pp, void *cuda_stream) {
    if (int rc = validate_fwd(pp)) return rc;
    const mia_ss_params &p = *pp;
    DeviceInfo di;
    if (int rc = device_info(di)) return rc;
    FwdPlan f;
    if (int rc = plan_fwd(p, di, true, f)) return rc;
#ifdef MIA_DEBUG
    char line[256];
    describe(f, line, sizeof(line));
    MIA_TRACE("fwd: %s", line);
#endif
    cudaStream_t stream = (cudaStream_t)cuda_stream;
    const bool of32 = p.otype == MIA_F32 && p.itype != MIA_F32;
    const cudaError_t rc = dispatch(p.itype, [&](auto *tag) {
        using T = typename std::remove_pointer<decltype(tag)>::type;
        switch (f.family) {
            case kCw: return mia::launch_fwd_cw<T>(f.tm, f.cw, f.grid, of32, stream);
            case kChunks: return mia::launch_fwd_chunks<T>(f.chunks, f.grid, of32, stream);
            case kRows: return mia::launch_fwd_rows<T>(f.rows, f.grid, of32, stream);
            case kStream: return mia::launch_fwd_stream<T>(f.stream, f.grid, of32, stream);
            case kRowsN: return mia::launch_fwd_rowsn<T>(f.rowsn, f.grid, of32, stream);
            default: return mia::launch_fwd_any<T>(f.ws, f.grid, stream);
        }
    });
    if (rc != cudaSuccess) return fail(MIA_ECUDA, "selective_scan_fwd (%s kernel) launch: %s", kFamilyName[f.family], cudaGetErrorString(rc));
    g_launches.fetch_add(f.launches());
    return MIA_OK;
}

size_t mia_selective_scan_bwd_workspace(const mia_ss_params *pp) {
    if (!pp) return 0;
    if (validate_sizes(*pp) != MIA_OK) return 0;     // sizes that the backward itself would reject
    DeviceInfo di;
    if (device_info(di) != MIA_OK) { di.sms = 148; di.smem_optin = 232448; }
    Plan pl;
    mia::ScanArgs a;
    if (plan_and_layout(*pp, di, true, pl, a) != MIA_OK) return 0;
    return workspace_layout(*pp, pl, di.sms).total;
}

int mia_selective_scan_bwd(const mia_ss_params *pp, void *cuda_stream) {
    if (int rc = validate_bwd(pp)) return rc;
    const mia_ss_params &p = *pp;
    DeviceInfo di;
    if (int rc = device_info(di)) return rc;
    BwdPlan b;
    if (int rc = plan_bwd(p, di, true, b)) return rc;
#ifdef MIA_DEBUG
    char line[256];
    describe(b, line, sizeof(line));
    MIA_TRACE("bwd: %s", line);
#endif
    const mia::ScanArgs &a = b.ws;
    cudaStream_t stream = (cudaStream_t)cuda_stream;
    if (b.atomic) {
        MIA_CUDA(cudaMemsetAsync(a.acc_dB, 0, b.w.acc_bytes, stream));
        MIA_CUDA(cudaMemsetAsync(a.acc_dC, 0, b.w.acc_bytes, stream));
        g_launches.fetch_add(2);
    }
    const bool of32 = p.otype == MIA_F32 && p.itype != MIA_F32;
    cudaError_t rc = dispatch(p.itype, [&](auto *tag) {
        using T = typename std::remove_pointer<decltype(tag)>::type;
        switch (b.family) {
            case kCw: return mia::launch_bwd_cw<T>(b.tm, b.cw, b.grid, of32, stream);
            case kRowsN: return mia::launch_bwd_rowsn<T>(b.rowsn, b.grid, of32, stream);
            case kRows: return mia::launch_bwd_rows<T>(b.rows, b.grid, of32, stream);
            default: return mia::launch_bwd_any<T>(a, b.grid, stream);
        }
    });
    if (rc != cudaSuccess) return fail(MIA_ECUDA, "selective_scan_bwd (%s kernel) launch: %s", kFamilyName[b.family], cudaGetErrorString(rc));
    g_launches.fetch_add(1);

    FinArgs f;
    memset(&f, 0, sizeof(f));
    f.batch = p.batch; f.dim = p.dim; f.L = p.seqlen; f.N = p.dstate; f.G = p.n_groups; f.delta_dim = p.delta_dim;
    f.ratio = p.dim / p.delta_dim; f.tiles = b.parts; f.bc_atomic = b.atomic; f.Lp = (p.seqlen + 3) & ~3;
    if (b.family == kRowsN) { f.oct_per_cta = b.rowsn.oct_per_cta; f.oct_per_group = b.rowsn.oct_per_group; }
    f.part_dA = a.part_dA; f.part_dD = a.part_dD; f.part_dbias = a.part_dbias; f.acc_dB = a.acc_dB; f.acc_dC = a.acc_dC;
    f.ddelta_full = a.ddelta_full;
    f.dA = p.dA; f.dD = p.dD; f.dbias = p.ddelta_bias; f.dB = p.dB; f.dC = p.dC; f.ddelta = p.ddelta;
    f.dA_ds = p.dA_d_stride; f.dA_ns = p.dA_dstate_stride;
    f.dB_bs = p.dB_batch_stride; f.dB_gs = p.dB_group_stride; f.dB_ns = p.dB_dstate_stride;
    f.dC_bs = p.dC_batch_stride; f.dC_gs = p.dC_group_stride; f.dC_ns = p.dC_dstate_stride;
    f.dd_bs = p.ddelta_batch_stride; f.dd_ds = p.ddelta_d_stride;
    f.n_bc = (long long)p.batch * p.n_groups * p.dstate * p.seqlen;
    f.n_dA = (long long)p.dim * p.dstate;
    f.n_dD = p.D ? p.dim : 0;
    f.n_db = p.delta_bias ? p.delta_dim : 0;
    f.n_dd = f.ratio > 1 ? (long long)p.batch * p.delta_dim * p.seqlen : 0;
    const long long total = (2 * f.n_bc + f.n_dd + 31) / 32 * 32 + 32 * (f.n_dA + f.n_dD + f.n_db);
    long long blocks = (total + 255) / 256;
    if (blocks > di.sms * 8) blocks = di.sms * 8;
    rc = dispatch(p.itype, [&](auto *tag) {
        using T = typename std::remove_pointer<decltype(tag)>::type;
        ss_finalize_kernel<T><<<(int)blocks, 256, 0, stream>>>(f);
        return cudaGetLastError();
    });
    if (rc != cudaSuccess) return fail(MIA_ECUDA, "selective_scan_bwd finalize launch: %s", cudaGetErrorString(rc));
    g_launches.fetch_add(1);
    return MIA_OK;
}

}  // extern "C"
