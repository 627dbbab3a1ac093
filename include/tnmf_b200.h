/*
 * tnmf_b200 -- C-ABI of the B200 (sm_100a) kernels for the shift-invariant NMF multiplicative-update
 * iteration of emdgroup/tnmf.
 *
 * This is the drop-in boundary: the entry points are what a `tnmf.backends.B200_Backend` binds (ctypes,
 * see INTEGRATION.md) to serve the reference's backend interface
 *     tnmf/backends/_Backend.py:35-130   (initialize / reconstruct / reconstruction_gradient_{H,W} /
 *                                         reconstruction_energy / normalize / convolve_multi_1d)
 * and the update arithmetic the reference facade applies to the backend's results
 *     tnmf/TransformInvariantNMF.py:217-271  (_multiplicative_update, _update_W, _update_H).
 *
 * Conventions
 *   - every pointer is a DEVICE pointer into memory owned by the caller (PyTorch owns all buffers); the
 *     library never allocates or frees user-visible memory; scratch is a caller-provided workspace whose
 *     size is reported by tnmf_workspace_bytes();
 *   - every call is stream-ordered on `stream` (a cudaStream_t passed as void*); nothing synchronises;
 *   - tensors are C-contiguous in the reference's layouts  V,R[n,c,*D]  W[m,c,*A]  H[n,m,*T]  except that H
 *     may carry arbitrary strides on its two leading axes (tnmf/backends/_Backend.py:124-125 passes
 *     H[:, i:i+1]) and a padded pitch between its rows (the stride of the second-to-last shift axis; the
 *     TMA kernels need every H stride to be a multiple of 4 elements);
 *   - the element type of all tensors is `dtype` (float or double; "dtype follows V",
 *     tnmf/backends/_Backend.py:92,95);
 *   - return value: 0 on success, a TNMF_E* code otherwise; errors never cross the boundary as exceptions.
 *     There is no CPU fallback: an unsupported request is an error.
 */
#ifndef TNMF_B200_H
#define TNMF_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TNMF_ABI_VERSION 6
#define TNMF_MAX_SHIFT_DIMS 3

/* element types */
#define TNMF_F32 0
#define TNMF_F64 1

/* reconstruction modes, tnmf/backends/_Backend.py:60-73 and tnmf/backends/_PyTorchBackend.py:42-52 */
#define TNMF_VALID    0   /* T = D + A - 1, no padding of H            */
#define TNMF_FULL     1   /* T = D - A + 1, H zero-padded (p, p)        */
#define TNMF_CIRCULAR 2   /* T = D,         H wrapped     (p, 0)        */

/* kernel family selection (diagnostics / tests); 0 lets the library choose */
#define TNMF_PATH_AUTO    0
#define TNMF_PATH_GENERIC 1   /* one-thread-per-output kernels, any rank <= 3, float and double */
#define TNMF_PATH_TILED   2   /* cp.async-staged register-tiled FP32-FMA kernels (rank <= 2, float, all modes) */
#define TNMF_PATH_TMA     3   /* persistent warp-specialised TMA + mbarrier kernels (rank 2, float, valid/full; also
                               * single-channel rank-1 batches, which run as one 2-D image of signal rows) */
#define TNMF_PATH_TC      4   /* tcgen05 3xTF32 tensor-core kernels with TMEM accumulators (reconstruction, H gradient /
                                 update, W gradient: rank 2, float, valid/full, atom height <= 15, C * atom width <= 64;
                                 reconstruction: C <= 4, atoms <= 64); operations / shapes without one use the TMA family.
                                 Rank 3 (float, valid): the same kernels over (sample, z-plane) pairs - reconstruction
                                 and W gradient one launch per atom plane, the H update with the atom planes as channels
                                 (C * A_z * A_x <= 64); reconstruction C <= 2, W gradient C * A_x <= 16, generic otherwise */

/* tnmf_problem.flags: switches of the 'auto' family choice (diagnostics / tests; 0 = the library's defaults).  They are part
 * of the problem description so that every behaviour of the library is reproducible through this interface alone. */
#define TNMF_FLAG_NO_ROWS_VIEW     1   /* single-channel rank-1 batches keep the rank-1 kernels */
#define TNMF_FLAG_ROWS_VIEW_ALWAYS 2   /* ... or run as one 2-D image of signal rows whatever the batch size (default: from
                                        * 2^20 signal elements on) */
#define TNMF_FLAG_NO_TC_HUPD       4   /* 'auto' keeps the H gradient / update off the tensor-core kernels */
#define TNMF_FLAG_NO_TC_RECON      8   /* ... the reconstruction */
#define TNMF_FLAG_NO_TC_GRADW     16   /* ... the W gradient */
#define TNMF_FLAG_NO_TC           28   /* all three */
#define TNMF_FLAG_NO_TMA          32   /* 'auto' skips the TMA family (cp.async tiled kernels instead) */
#define TNMF_FLAG_NO_TMEM_OPERAND 64   /* tensor-core kernels keep their expanded operand in shared memory (the round-1
                                        * kernels) instead of tensor memory */

/* operations, for tnmf_kernel_family() */
#define TNMF_OP_RECONSTRUCT 0
#define TNMF_OP_GRADIENT_H  1   /* also the fused H update */
#define TNMF_OP_GRADIENT_W  2

/* status codes */
#define TNMF_OK            0
#define TNMF_EINVAL        1   /* malformed problem description / null pointer                     */
#define TNMF_EUNSUPPORTED  2   /* valid request the library has no kernel for (Python: NotImplementedError) */
#define TNMF_EWORKSPACE    3   /* workspace too small                                              */
#define TNMF_ECUDA      1000   /* TNMF_ECUDA + cudaError_t                                         */

/* Geometry of one factorisation problem.  Shift axes are listed slowest first, exactly as in the shapes of
 * the reference tensors; unused trailing entries are ignored. */
typedef struct tnmf_problem {
    int32_t ndim;                               /* number of shift axes, 1..3                        */
    int32_t dtype;                              /* TNMF_F32 / TNMF_F64                               */
    int32_t mode;                               /* TNMF_VALID / TNMF_FULL / TNMF_CIRCULAR            */
    int32_t path;                               /* TNMF_PATH_*                                       */
    int32_t n_samples;                          /* N (of this call: a minibatch passes its own size) */
    int32_t n_channels;                         /* C                                                 */
    int32_t n_atoms;                            /* M                                                 */
    int32_t h_pitch;                            /* element stride between rows of H; 0 = dense (T[-1]) */
    int32_t sample_shape[TNMF_MAX_SHIFT_DIMS];  /* D                                                 */
    int32_t atom_shape[TNMF_MAX_SHIFT_DIMS];    /* A                                                 */
    int64_t h_stride_n;                         /* element strides of H's axes 0 and 1; 0 = contiguous */
    int64_t h_stride_m;
    int32_t flags;                              /* TNMF_FLAG_* (0 = defaults)                        */
    int32_t reserved;                           /* must be 0                                         */
} tnmf_problem;

int         tnmf_abi_version(void);
const char *tnmf_status_string(int status);

/* Extent of H along the shift axes.  Replaces Backend._n_transforms, tnmf/backends/_Backend.py:60-73. */
int tnmf_transform_shape(const tnmf_problem *p, int32_t *t_shape /* [ndim] */);

/* Bytes of scratch the calls below need for this problem (pre-arranged atom slices, split-K partials of the
 * W gradient, per-block energy partials).  Always a multiple of 256; the workspace must be 256-byte aligned.
 * The calls of one problem may share one workspace as long as they are ordered on one stream. */
size_t tnmf_workspace_bytes(const tnmf_problem *p);

/* 1 if shared-memory staged FP32 kernels (TMA or cp.async) serve this problem, 0 if the generic kernels do. */
int tnmf_uses_tiled_path(const tnmf_problem *p);

/* The TNMF_PATH_* family that serves operation `op` (TNMF_OP_*) of this problem, or -1 if the problem is malformed /
 * the forced `path` cannot serve it. */
int tnmf_kernel_family(const tnmf_problem *p, int op);

/* Name of the hot kernel that serves operation `op` of this problem ("recon_ts_kernel", "hupd_tma_kernel", ...; the
 * __global__ function an ncu launch list shows), or "none" like tnmf_kernel_family's -1.  Static string.  Diagnostics:
 * parity tests and bench.py record which kernel they exercised. */
const char *tnmf_kernel_name(const tnmf_problem *p, int op);

/* How many kernels one call of operation `op` launches for this problem (the fused / unfused H operations alike), or -1
 * like tnmf_kernel_family.  Bookkeeping for callers that report launch counts (bench.py's "gpu_launches"). */
int tnmf_launch_count(const tnmf_problem *p, int op);

/* R[n,c,d] = sum_m sum_a W[m,c,a] * Hpad[n,m,d+p-a].
 * Replaces Backend.reconstruct, tnmf/backends/_Backend.py:120-122 (NumPy.py:122-132, PyTorch.py:26-43). */
int tnmf_reconstruct(const tnmf_problem *p, const void *W, const void *H, void *R, void *workspace,
                     size_t workspace_bytes, void *stream);

/* *energy (a double in device memory) = 0.5 * sum (V - reconstruct(W,H))^2, reduced on the device; if R is
 * non-null the reconstruction is stored as well.
 * Replaces Backend.reconstruction_energy, tnmf/backends/_Backend.py:127-130. */
int tnmf_reconstruct_energy(const tnmf_problem *p, const void *V, const void *W, const void *H, void *R,
                            double *energy, void *workspace, size_t workspace_bytes, void *stream);

/* neg[n,m,t] = sum_c sum_a W[m,c,a] * V[n,c,t-p+a],  pos likewise from R (mode-specific adjoint padding).
 * R must hold reconstruct(W,H).  neg and pos are contiguous [n,m,*T].
 * Replaces Backend.reconstruction_gradient_H, tnmf/backends/_Backend.py:110-118 (NumPy.py:93-120). */
int tnmf_gradient_h(const tnmf_problem *p, const void *V, const void *R, const void *W,
                    void *neg, void *pos, void *workspace, size_t workspace_bytes, void *stream);

/* Fused H update: the two correlations above plus, in the epilogue and in the reference's order of
 * roundings,   pos += lambda * (G - H);  pos += lambda_cross * (Gsum - G);  pos += reg;  H = (H*neg)/pos
 * where G = convolve_multi_1d(H, inhibition kernels) (may be null when lambda == lambda_cross == 0),
 * Gsum[n,1,t] = sum_m G (may be null when lambda_cross == 0), reg = eps + sparsity and lambda_cross is
 * already divided by (n_atoms - 1).  H is updated in place.
 * Replaces TransformInvariantNMF._update_H + _multiplicative_update,
 * tnmf/TransformInvariantNMF.py:217-235,246-271. */
int tnmf_update_h(const tnmf_problem *p, const void *V, const void *R, const void *W, void *H,
                  double reg, const void *G, double lambda, const void *Gsum, double lambda_cross,
                  void *workspace, size_t workspace_bytes, void *stream);

/* neg[m,c,a] = sum_n sum_d Hpad[n,m,d+p-a] * V[n,c,d],  pos likewise from R (R must hold reconstruct(W,H)).
 * Split-K over samples and positions into per-block partials in `workspace`, then a fixed-order
 * (deterministic) final reduction in double.
 * Replaces Backend.reconstruction_gradient_W, tnmf/backends/_Backend.py:100-108 (NumPy.py:69-91). */
int tnmf_gradient_w(const tnmf_problem *p, const void *V, const void *R, const void *H,
                    void *neg, void *pos, void *workspace, size_t workspace_bytes, void *stream);

/* Plane windows: tnmf_update_h / tnmf_gradient_w restricted to the activation indices t in [t_lo, t_hi) along the FIRST
 * shift axis (z-planes of a volume, rows of an image, positions of a signal).  The H update writes H only inside the
 * window (it reads H, V and R wherever the correlations need them); the W gradient sums over the window only, as if H
 * were zero outside it.  A band of a halo-sharded fit (tnmf_b200/halo.py) uses them to skip its halo planes, which the
 * next exchange overwrites and which belong to the neighbours' share of the W gradient.  0 <= t_lo <= t_hi <= T[0] (else
 * TNMF_EINVAL); the full window [0, T[0]) gives results bitwise equal to the unwindowed calls.
 * Served by the plane mode of the tensor-core kernels (three shift axes, float32, 'valid') and by the generic kernels
 * (any rank, mode and dtype); problems that another family serves return TNMF_EUNSUPPORTED.  tnmf_kernel_family and
 * tnmf_kernel_name of the problem name the kernels a windowed call runs; tnmf_workspace_bytes and tnmf_launch_count of
 * the problem bound what it needs and launches (the W gradient skips the per-atom-plane launches whose sample planes
 * all lie outside the window). */
int tnmf_update_h_planes(const tnmf_problem *p, const void *V, const void *R, const void *W, void *H,
                         double reg, const void *G, double lambda, const void *Gsum, double lambda_cross,
                         int32_t t_lo, int32_t t_hi, void *workspace, size_t workspace_bytes, void *stream);
int tnmf_gradient_w_planes(const tnmf_problem *p, const void *V, const void *R, const void *H,
                           void *neg, void *pos, int32_t t_lo, int32_t t_hi,
                           void *workspace, size_t workspace_bytes, void *stream);

/* W = (W * neg) / (pos + eps);  W[m,c,:] /= sum_a W[m,c,a].  In place; neg/pos are left untouched.
 * Replaces TransformInvariantNMF._update_W's arithmetic, tnmf/TransformInvariantNMF.py:217-244, and
 * Backend.normalize, tnmf/backends/_Backend.py:75-77. */
int tnmf_update_w(const tnmf_problem *p, void *W, const void *neg, const void *pos, double eps, void *stream);

/* Multi-GPU W step in ONE kernel over NVLink peer memory: the stacked W gradient grad = [neg; pos] of this rank is summed
 * with those of all `world` ranks and the W update above is applied to the sum - the all-reduce that the sample-sharded
 * iteration needs (the sum over sample blocks of Cyclic_MU, tnmf/TransformInvariantNMF.py:457-465) fused with
 * tnmf/TransformInvariantNMF.py:217-244 and Backend.normalize, tnmf/backends/_Backend.py:75-77.
 *   buffers[r]   rank r's symmetric exchange buffer mapped into THIS process (tnmf_peer_buffer_bytes bytes each, zeroed
 *                once before the first call, identical layout on every rank); every rank calls with the same world,
 *   state        two zero-initialised uint32 in this rank's device memory (epoch, block counter),
 * Collective: every rank must make the same sequence of calls.  The ranks add the same numbers in the same (rank) order
 * in double, so W stays bit-identical on all ranks.  The call is stream-ordered and may be captured into a CUDA graph. */
#define TNMF_MAX_PEERS 16
typedef struct tnmf_peer_world {
    int32_t world, rank;
    void *buffers[TNMF_MAX_PEERS];
} tnmf_peer_world;
size_t tnmf_peer_buffer_bytes(const tnmf_problem *p, int32_t world);
int tnmf_allreduce_update_w(const tnmf_problem *p, void *W, const void *grad, const tnmf_peer_world *peers, void *state,
                            double eps, void *stream);

/* arr[o,:,i] /= sum over the middle axis, for a tensor viewed as [outer, len, inner].
 * Replaces Backend.normalize, tnmf/backends/_Backend.py:75-77, for contiguous reduction axes. */
int tnmf_normalize(int32_t dtype, void *arr, int64_t outer, int64_t len, int64_t inner, void *stream);

/* out = in convolved along one axis with a centred odd kernel, zero boundary.  The tensor is viewed as
 * [outer, len, inner]; `taps` are n_taps doubles in device memory.  in != out.
 * Replaces one pass of Backend.convolve_multi_1d, tnmf/backends/_NumPyBackend.py:56-64. */
int tnmf_convolve_1d(int32_t dtype, const void *in, void *out, int64_t outer, int64_t len, int64_t inner,
                     const double *taps, int32_t n_taps, void *stream);

/* Gsum[n,0,t] = sum_m G[n,m,t] for contiguous G[n,m,inner].
 * Replaces `inhibition_gradient.sum(axis=1, keepdims=True)`, tnmf/TransformInvariantNMF.py:263. */
int tnmf_sum_atoms(int32_t dtype, const void *G, void *Gsum, int64_t n_samples, int64_t n_atoms,
                   int64_t inner, void *stream);

/* Throughput probe used by bench.py for the FP32-pipe roofline denominator: launches a dependent-free FFMA
 * loop on every SM and writes the elapsed-independent checksum to `sink` (>= 4 bytes).  `flops_out` (host)
 * receives the number of floating-point operations the launch performs. */
int tnmf_fp32_peak_probe(void *sink, int32_t iterations, double *flops_out, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* TNMF_B200_H */
