/* C ABI of the B200-native selective scan (libmia_scan.so).
 *
 * This is the drop-in boundary for the reference's native op
 *   selective_scan_cuda_oflex.fwd / .bwd
 *     (R2GenCSR/VMamba/kernels/selective_scan/csrc/selective_scan/cusoflex/selective_scan_oflex.cpp:143-231, 233-355,
 *      pybind at :357-360),
 *   selective_scan_cuda_core.fwd / .bwd   (.../cus/selective_scan.cpp:157-164, 241-250)  == oflex with otype == itype,
 *   and the mamba_ssm signature with the z gate, selective_scan_cuda.fwd / .bwd, as called at
 *     R2GenCSR/VMamba/classification/models/vmamba.py:255, 266-269 and
 *     CXPMRG_Bench_MambaXray_VL/arm/Finetuning/mamba_simple.py:693-704 (through mamba_ssm's selective_scan_fn).
 *
 * Plain pointers and sizes only: the caller (any host language) owns every buffer, the library
 * only launches kernels on the stream it is given.  All pointers are DEVICE pointers.  Strides are in
 * ELEMENTS (like SSMParamsBase, selective_scan_oflex.h:27-60); the innermost (sequence) stride of
 * u, delta, z, B, C, out, dout, du, ddelta, dz, dB, dC must be 1 (selective_scan_oflex.cpp:167-168,186,188).
 *
 * Every entry point returns 0 on success or a negative MIA_E* code; mia_last_error() returns a
 * thread-local message for the last failure (the Python binding raises RuntimeError with it, mirroring
 * TORCH_CHECK -> RuntimeError in the reference).  Calls are asynchronous w.r.t. the host and reentrant.
 */
#ifndef MIA_SELECTIVE_SCAN_H_
#define MIA_SELECTIVE_SCAN_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MIA_ABI_VERSION 2

enum { MIA_F32 = 0, MIA_F16 = 1, MIA_BF16 = 2 };

enum {
    MIA_OK = 0,
    MIA_EINVAL = -1,     /* bad shape / dtype / stride / null pointer (the reference's TORCH_CHECKs) */
    MIA_ECUDA = -2,      /* a CUDA runtime call or the launch failed */
    MIA_EWORKSPACE = -3  /* workspace missing or too small */
};

typedef struct mia_ss_params {
    /* ---- sizes (selective_scan_oflex.cpp:169-180) */
    int32_t batch, dim, seqlen, dstate, n_groups, delta_dim;
    int32_t itype;           /* dtype of u, delta, B, C, z and of du, ddelta, dB, dC, dz */
    int32_t otype;           /* dtype of out/out_z (fwd) and of dout/out_saved (bwd): itype or MIA_F32 ("oflex") */
    int32_t delta_softplus;  /* 0/1 */
    int32_t n_chunks;        /* 3rd dim of x; must equal mia_ss_num_chunks(seqlen) */

    /* ---- inputs */
    const void *u;           /* (batch, dim, seqlen)            itype */
    const void *delta;       /* (batch, delta_dim, seqlen)      itype; dim % delta_dim == 0 */
    const void *A;           /* (dim, dstate)                   f32, any strides */
    const void *B;           /* (batch, n_groups, dstate, seqlen) itype */
    const void *C;           /* same */
    const void *D;           /* (dim) f32 contiguous, or NULL */
    const void *delta_bias;  /* (delta_dim) f32 contiguous, or NULL */
    const void *z;           /* (batch, dim, seqlen) itype, or NULL (mamba_ssm gate: out_z = out * silu(z)) */
    int64_t u_batch_stride, u_d_stride;
    int64_t delta_batch_stride, delta_d_stride;
    int64_t A_d_stride, A_dstate_stride;
    int64_t B_batch_stride, B_group_stride, B_dstate_stride;
    int64_t C_batch_stride, C_group_stride, C_dstate_stride;
    int64_t z_batch_stride, z_d_stride;

    /* ---- forward outputs */
    void *out;               /* (batch, dim, seqlen) otype : y + D*u (before the gate) */
    void *out_z;             /* (batch, dim, seqlen) otype, required iff z != NULL */
    float *x;                /* (batch, dim, n_chunks, 2*dstate) f32 contiguous: per-chunk (prod a, h) checkpoints;
                                x[:, :, -1, 1::2] is the last state (test_selective_scan.py:79). Written by fwd,
                                read by bwd when n_chunks > 1. */
    int64_t out_batch_stride, out_d_stride;
    int64_t out_z_batch_stride, out_z_d_stride;

    /* ---- backward inputs */
    const void *dout;        /* (batch, dim, seqlen) otype: grad of out (z == NULL) or of out_z (z != NULL) */
    const void *out_saved;   /* fwd `out`, otype; required iff z != NULL */
    int64_t dout_batch_stride, dout_d_stride;
    int64_t out_saved_batch_stride, out_saved_d_stride;

    /* ---- backward outputs (all fully overwritten, no pre-zeroing needed) */
    void *du;                /* (batch, dim, seqlen) itype */
    void *ddelta;            /* (batch, delta_dim, seqlen) itype (already summed over the delta group) */
    float *dA;               /* (dim, dstate) f32 */
    void *dB, *dC;           /* (batch, n_groups, dstate, seqlen) itype */
    float *dD;               /* (dim) f32, required iff D != NULL */
    float *ddelta_bias;      /* (delta_dim) f32, required iff delta_bias != NULL */
    void *dz;                /* (batch, dim, seqlen) itype, required iff z != NULL */
    int64_t du_batch_stride, du_d_stride;
    int64_t ddelta_batch_stride, ddelta_d_stride;
    int64_t dA_d_stride, dA_dstate_stride;
    int64_t dB_batch_stride, dB_group_stride, dB_dstate_stride;
    int64_t dC_batch_stride, dC_group_stride, dC_dstate_stride;
    int64_t dz_batch_stride, dz_d_stride;

    /* ---- scratch for the deterministic reductions of the backward (f32 partials) */
    void *workspace;
    size_t workspace_bytes;

    /* ---- (ABI 2) optional block states handed from fwd to the matching bwd: mia_ss_block_state_floats(p) floats, 128-byte
     * aligned, or NULL.  The d_state == 1 column-walk forward (csrc/scan_fwd_cw.cuh) writes the state entering every group of
     * 16 tokens of every row here (when mia_ss_fwd_writes_block_states(p) != 0; the layout is the kernel pair's own, see
     * that file); given to the backward of the SAME inputs it lets the column-walk backward (csrc/scan_bwd_cw.cuh) skip
     * the forward recompute pass.  NULL on either side = the resident-row / warp-scan kernels, same results. */
    float *hblk;
} mia_ss_params;

/* ABI / build identification. */
int mia_abi_version(void);
const char *mia_last_error(void);

/* Checkpoint geometry: tokens per chunk for a sequence length, and ceil(seqlen / chunk). */
int mia_ss_chunk_len(int seqlen);
int mia_ss_num_chunks(int seqlen);

/* Block states (see mia_ss_params.hblk): size in floats for these sizes, and whether the forward for exactly these
 * parameters (pointers, strides, dtypes) will fill p->hblk (0 when the shape takes a kernel that does not produce them). */
size_t mia_ss_block_state_floats(const mia_ss_params *p);
int mia_ss_fwd_writes_block_states(const mia_ss_params *p);

/* Forward.  Replaces selective_scan_fwd (selective_scan_oflex.cpp:143-231). */
int mia_selective_scan_fwd(const mia_ss_params *p, void *cuda_stream);

/* Bytes of workspace the backward needs for these sizes (only sizes/dtypes/optional-pointer presence are read). */
size_t mia_selective_scan_bwd_workspace(const mia_ss_params *p);

/* Backward.  Replaces selective_scan_bwd (selective_scan_oflex.cpp:233-355) including its post-kernel
 * casts (:347) and delta-group folds (:348-353). */
int mia_selective_scan_bwd(const mia_ss_params *p, void *cuda_stream);

/* Which kernel mia_selective_scan_fwd (backward = 0) / _bwd (backward = 1) would launch for *p, and its geometry, as one
 * line of space-separated key=value pairs starting with "kernel=". sms / smem_optin describe the device (<= 0: query the
 * current device); when both are given no CUDA call is made. Tensor maps are not encoded (assumed encodable).
 * Validates *p like the call itself (the backward's workspace included) and returns the same error codes. */
int mia_ss_describe_plan(const mia_ss_params *p, int backward, int sms, int smem_optin, char *buf, size_t buf_len);

/* CrossScan / CrossMerge of SS2D (R2GenCSR/VMamba/classification/models/vmamba.py:25-67, csm_triton.py:163-235).
 * x, y: (batch, channels, H, W) contiguous; xs, ys: (batch, 4, channels, H*W) contiguous; same dtype in and out.
 * scan: xs[:,0] = row-major, xs[:,1] = column-major, xs[:,2:4] = their reversals.  merge = its adjoint (fp32 sum).
 * Any H, W: planes are staged in shared memory while one fits (H W <= ~50 K elements), gathered directly beyond. */
int mia_cross_scan(const void *x, void *xs, int batch, int channels, int H, int W, int dtype, void *cuda_stream);
int mia_cross_merge(const void *ys, void *y, int batch, int channels, int H, int W, int dtype, void *cuda_stream);
const char *mia_cs_last_error(void);   /* message of the last failed mia_cross_scan / mia_cross_merge / mia_silu_gate on this thread */

/* out_z[i] = out[i] * silu(z[i]) over n contiguous elements (fp32 arithmetic): the gate of the mamba_ssm signature recomputed
 * from the saved pre-gate output -- selective_scan_cuda.bwd(..., recompute_out_z=True), test_selective_scan.py:105-108. */
int mia_silu_gate(const void *out, const void *z, void *out_z, long long n, int z_dtype, int out_dtype, void *cuda_stream);

/* Depth-wise causal conv1d (+ bias, + SiLU) of the Mamba mixers: y[b, d, t] = act(bias[d] + sum_k w[d, k] x[b, d, t - (K-1) + k]).
 * Replaces causal_conv1d.causal_conv1d_fn (un-vendored; call sites arm/Finetuning/mamba_simple.py:676-681 of the three ARM sub-projects) == the in-repo
 * fallback `self.act(self.conv1d(x)[..., :seqlen])` (:112-120, 673).  x, y, dy, dx: (batch, dim, seqlen), sequence stride 1,
 * batch / channel strides in elements (multiples of 4; x is usually the first half of xz); weight (dim, width <= 4) and
 * bias (dim, may be NULL) fp32 contiguous; seqlen % 4 == 0.  bwd writes dx, dweight (dim, width) and dbias (dim, if not
 * NULL) completely (deterministic, no atomics).  mia_conv_last_error() holds the message of the last failure. */
int mia_causal_conv1d_fwd(const void *x, const float *weight, const float *bias, void *y, int batch, int dim, int seqlen, int width,
                          int silu, int dtype, long long x_batch_stride, long long x_d_stride, long long y_batch_stride,
                          long long y_d_stride, void *cuda_stream);
int mia_causal_conv1d_bwd(const void *x, const float *weight, const float *bias, const void *dy, void *dx, float *dweight, float *dbias,
                          int batch, int dim, int seqlen, int width, int silu, int dtype, long long x_batch_stride, long long x_d_stride,
                          long long dy_batch_stride, long long dy_d_stride, long long dx_batch_stride, long long dx_d_stride,
                          void *cuda_stream);
const char *mia_conv_last_error(void);

/* Depth-wise 3x3 conv2d (stride 1, padding 1, + bias, + SiLU) of SS2D on channel-first activations:
 * `self.act(self.conv2d(x))`, R2GenCSR/VMamba/classification/models/vmamba.py:574-582, 1120-1122.  x, y, dy, dx: (batch,
 * channels, H, W) contiguous, H*W <= 16384; weight (channels, 9) and bias (channels, may be NULL) fp32.  bwd writes dx,
 * dweight (channels, 9) and dbias (if not NULL) completely (deterministic, no atomics). */
int mia_dwconv2d_fwd(const void *x, const float *weight, const float *bias, void *y, int batch, int channels, int H, int W, int silu,
                     int dtype, void *cuda_stream);
int mia_dwconv2d_bwd(const void *x, const float *weight, const float *bias, const void *dy, void *dx, float *dweight, float *dbias,
                     int batch, int channels, int H, int W, int silu, int dtype, void *cuda_stream);
const char *mia_dwconv2d_last_error(void);

/* Number of selective-scan kernel launches issued by this library in this process since load (bench.py gpu_launches). */
uint64_t mia_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* MIA_SELECTIVE_SCAN_H_ */
