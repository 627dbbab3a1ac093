// Shared definitions of the tnmf_b200 kernels (sm_100a).
//
// Internally every problem is three-dimensional (z, y, x); lower ranks get leading extents of 1.  The three
// reconstruction modes of the reference (tnmf/backends/_Backend.py:60-73, _PyTorchBackend.py:42-52) differ
// only in an index offset and a boundary rule, so one set of kernels serves all of them:
//
//   R[d]      = sum_a W[a] * Hext[d + off - a]          Hext: H on [0,T), else 0 ('wrap': periodic)
//   gradH[t]  = sum_a W[a] * Xext[t - off + a]          Xext: X on [0,D), else 0 ('wrap': periodic)
//   gradW[a]  = sum_d Hext[d + off - a] * X[d]
//
//   valid: off = A-1, T = D+A-1 (boundary rule never triggers for H)
//   full:  off = 0,   T = D-A+1 (zero rule for H, never triggers for X)
//   circular: off = 0, T = D, wrap
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "../../include/tnmf_b200.h"

namespace tnmf {

struct Geo {
    int N, C, M;
    int D[3];      // sample extent  (z, y, x)
    int A[3];      // atom extent
    int T[3];      // activation extent
    int off[3];    // A-1 for 'valid', 0 otherwise
    int wrap;      // 1 for 'circular'
    int ndim;
    long long hsn, hsm;   // element strides of H's leading axes
    long long hsy;        // element stride between rows of H (>= T[2]; the last axis is always dense)
    int flags;            // tnmf_problem.flags (TNMF_FLAG_*)
};

__host__ __device__ inline long long vol3(const int *s) { return (long long)s[0] * s[1] * s[2]; }

// a third shift axis in use: the 2-D kernel families do not serve the problem (tc_common.cuh: plane mode)
inline bool plane_problem(const Geo &g) { return g.D[0] != 1 || g.A[0] != 1; }

// Map a logical index onto [0, extent): returns false when the element is an implicit zero.
__device__ __forceinline__ bool fold_index(int &i, int extent, int wrap) {
    if (wrap) {
        i %= extent;
        if (i < 0) i += extent;
        return true;
    }
    return (unsigned)i < (unsigned)extent;
}

inline int status_from_cuda(cudaError_t e) { return e == cudaSuccess ? TNMF_OK : TNMF_ECUDA + (int)e; }

#define TNMF_CHECK_LAUNCH()                                        \
    do {                                                           \
        cudaError_t e__ = cudaGetLastError();                      \
        if (e__ != cudaSuccess) return status_from_cuda(e__);      \
    } while (0)

// ---- implemented in generic_kernels.cu -----------------------------------------------------------------
template <typename T> int generic_reconstruct(const Geo &g, const T *W, const T *H, T *R, const T *V,
                                              double *energy_partials, int *n_partials, cudaStream_t st);
// t_lo, t_hi: the window of activation indices [t_lo, t_hi) along the first shift axis that is updated / correlated
// (t_hi < 0: all of them)
template <typename T> int generic_gradient_h(const Geo &g, const T *V, const T *R, const T *W, T *neg, T *pos,
                                             T *H, double reg, const T *G, double lambda, const T *Gsum,
                                             double lambda_cross, cudaStream_t st, int t_lo = 0, int t_hi = -1);
template <typename T> int generic_gradient_w(const Geo &g, const T *V, const T *R, const T *H, T *neg, T *pos,
                                             cudaStream_t st, int t_lo = 0, int t_hi = -1);
int generic_energy_partial_capacity(const Geo &g);

// ---- implemented in tiled_kernels.cu --------------------------------------------------------------------
bool tiled_supported(const Geo &g, int dtype);
size_t tiled_workspace_bytes(const Geo &g);
int tiled_reconstruct(const Geo &g, const float *W, const float *H, float *R, const float *V,
                      double *energy_partials, int *n_partials, cudaStream_t st);
int tiled_gradient_h(const Geo &g, const float *V, const float *R, const float *W, float *neg, float *pos,
                     float *H, double reg, const float *G, double lambda, const float *Gsum,
                     double lambda_cross, cudaStream_t st);
int tiled_gradient_w(const Geo &g, const float *V, const float *R, const float *H, float *neg, float *pos,
                     void *workspace, size_t workspace_bytes, cudaStream_t st);

// ---- implemented in tma_kernels.cu ------------------------------------------------------------------------
bool tma_recon_supported(const Geo &g, int dtype);
bool tma_hupd_supported(const Geo &g, int dtype);
bool tma_gradw_supported(const Geo &g, int dtype);
size_t tma_workspace_bytes(const Geo &g, int dtype);
double *tma_energy_partials(const Geo &g, void *workspace);
int tma_reconstruct(const Geo &g, const float *W, const float *H, float *R, const float *V, double *energy_partials,
                    int *n_partials, void *workspace, size_t workspace_bytes, cudaStream_t st);
int tma_gradient_h(const Geo &g, const float *V, const float *R, const float *W, float *neg, float *pos, float *H,
                   double reg, const float *G, double lambda, const float *Gsum, double lambda_cross, void *workspace,
                   size_t workspace_bytes, cudaStream_t st);
int tma_gradient_w(const Geo &g, const float *V, const float *R, const float *H, float *neg, float *pos,
                   void *workspace, size_t workspace_bytes, cudaStream_t st);

// ---- implemented in tc_hupd.cu (tcgen05 3xTF32) -------------------------------------------------------------
bool tc_hupd_supported(const Geo &g, int dtype);
int tc_hupd_launches(const Geo &g);
int tc_gradient_h(const Geo &g, const float *V, const float *R, const float *W, float *neg, float *pos, float *H,
                  double reg, const float *G, double lambda, const float *Gsum, double lambda_cross, cudaStream_t st);

// ---- implemented in tc_gradw.cu (tcgen05 3xTF32) ------------------------------------------------------------
bool tc_gradw_supported(const Geo &g, int dtype);
size_t tc_gradw_workspace_bytes(const Geo &g);
int tc_gradw_launches(const Geo &g);
int tc_gradient_w(const Geo &g, const float *V, const float *R, const float *H, float *neg, float *pos, void *workspace,
                  size_t workspace_bytes, cudaStream_t st);

// ---- implemented in tc_gradw_ts.cu (tcgen05 3xTF32, expanded operand in tensor memory) ------------------------
bool tc_gradw_ts_supported(const Geo &g, int dtype);
size_t tc_gradw_ts_workspace_bytes(const Geo &g);
int tc_gradw_ts_launches(const Geo &g);
int tc_gradient_w_ts(const Geo &g, const float *V, const float *R, const float *H, float *neg, float *pos, void *workspace,
                     size_t workspace_bytes, cudaStream_t st);

// ---- implemented in tc_gradw_ns.cu (tcgen05 3xTF32, narrow atoms: hi/lo, two rows and both tensors stacked in the lanes) --
bool tc_gradw_ns_supported(const Geo &g, int dtype);
size_t tc_gradw_ns_workspace_bytes(const Geo &g);
int tc_gradw_ns_launches(const Geo &g);
// t_lo, t_hi: 3-D only, correlate with the activation planes [t_lo, t_hi) only (t_hi < 0: all of them)
int tc_gradient_w_ns(const Geo &g, const float *V, const float *R, const float *H, float *neg, float *pos, void *workspace,
                     size_t workspace_bytes, cudaStream_t st, int t_lo = 0, int t_hi = -1);

// ---- implemented in tc_recon.cu (tcgen05 3xTF32) ------------------------------------------------------------
bool tc_recon_supported(const Geo &g, int dtype);
int tc_recon_partials(const Geo &g);
int tc_reconstruct(const Geo &g, const float *W, const float *H, float *R, const float *V, double *energy_partials,
                   int *n_partials, cudaStream_t st);

// ---- implemented in tc_hupd_ts.cu (tcgen05 3xTF32, expanded operand in tensor memory) ---------------------------
bool tc_hupd_ts_supported(const Geo &g, int dtype);
int tc_hupd_ts_launches(const Geo &g);
// t_lo, t_hi: 3-D only, update the activation planes [t_lo, t_hi) only (t_hi < 0: all of them)
int tc_gradient_h_ts(const Geo &g, const float *V, const float *R, const float *W, float *neg, float *pos, float *H,
                     double reg, const float *G, double lambda, const float *Gsum, double lambda_cross, cudaStream_t st,
                     int t_lo = 0, int t_hi = -1);

// ---- implemented in tc_recon_ts.cu (tcgen05 3xTF32, activation row ring in tensor memory) ---------------------
bool tc_recon_ts_supported(const Geo &g, int dtype);
int tc_recon_ts_partials(const Geo &g);
int tc_reconstruct_ts(const Geo &g, const float *W, const float *H, float *R, const float *V, double *energy_partials,
                      int *n_partials, cudaStream_t st);

// ---- implemented in tc_recon_os.cu (tcgen05 3xTF32, narrow atoms: output-row accumulator ring in tensor memory) -------
bool tc_recon_os_supported(const Geo &g, int dtype);
int tc_recon_os_partials(const Geo &g);
int tc_recon_os_launches(const Geo &g);          // one per atom plane
int tc_reconstruct_os(const Geo &g, const float *W, const float *H, float *R, const float *V, double *energy_partials,
                      int *n_partials, cudaStream_t st);

// ---- implemented in elementwise.cu ----------------------------------------------------------------------
int finish_energy(const double *partials, int n, double *energy, cudaStream_t st);
template <typename T> int finish_gradient_w(const T *partials, int n_partials, long long count, T *neg, T *pos,
                                            cudaStream_t st);
template <typename T> int update_w(const Geo &g, T *W, const T *neg, const T *pos, double eps, cudaStream_t st);
template <typename T> int normalize_axis(T *arr, long long outer, long long len, long long inner, cudaStream_t st);
template <typename T> int convolve_axis(const T *in, T *out, long long outer, long long len, long long inner,
                                        const double *taps, int n_taps, cudaStream_t st);
template <typename T> int sum_atoms(const T *G, T *Gsum, long long n, long long m, long long inner, cudaStream_t st);
int fp32_peak_probe(void *sink, int iterations, double *flops_out, cudaStream_t st);
int sm_count_cached();

// ---- implemented in peer_update_w.cu (all-reduce of the W gradient fused with the W update, NVLink peer memory) ------
size_t peer_buffer_bytes(const Geo &g, int dtype, int world);
template <typename T> int allreduce_update_w(const Geo &g, int dtype, T *W, const T *grad, const tnmf_peer_world *pw,
                                             unsigned *state, double eps, cudaStream_t st);

}  // namespace tnmf
