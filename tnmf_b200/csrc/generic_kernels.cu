// Generic kernels: one thread per output element (one block per output for the W gradient), any rank <= 3,
// all reconstruction modes, float and double.  They serve the shapes the register-tiled kernels do not
// (three shift axes, double precision) and are the in-device cross-check of the tiled path in the tests.
// Bound: FP32/FP64 FMA pipe with L1/L2-served operands; no shared-memory staging.
#include "common.cuh"

namespace tnmf {

static constexpr int kGenericThreads = 256;
static constexpr int kGenericMaxBlocks = 148 * 16;

int generic_energy_partial_capacity(const Geo &) { return kGenericMaxBlocks; }

template <typename T>
__device__ __forceinline__ double block_sum_double(double v, double *smem) {
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (lane == 0) smem[warp] = v;
    __syncthreads();
    if (warp == 0) {
        v = (lane < (blockDim.x >> 5)) ? smem[lane] : 0.0;
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    }
    return v;   // valid in thread 0
}

// R[n,c,d] = sum_m sum_a W[m,c,a] * Hext[n,m,d+off-a]      (tnmf/backends/NumPy.py:122-132)
template <typename T>
__global__ void __launch_bounds__(kGenericThreads)
generic_reconstruct_kernel(Geo g, const T *__restrict__ W, const T *__restrict__ H, T *__restrict__ R,
                           const T *__restrict__ V, double *__restrict__ energy_partials) {
    __shared__ double red[32];
    const long long dvol = vol3(g.D), avol = vol3(g.A);
    const long long total = (long long)g.N * g.C * dvol;
    double e_local = 0.0;
    for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
         idx += (long long)gridDim.x * blockDim.x) {
        long long r = idx;
        const int x = (int)(r % g.D[2]); r /= g.D[2];
        const int y = (int)(r % g.D[1]); r /= g.D[1];
        const int z = (int)(r % g.D[0]); r /= g.D[0];
        const int c = (int)(r % g.C);
        const int n = (int)(r / g.C);
        T acc = 0;
        for (int m = 0; m < g.M; ++m) {
            const T *w = W + ((long long)m * g.C + c) * avol;
            const T *h = H + n * g.hsn + m * g.hsm;
            for (int az = 0; az < g.A[0]; ++az) {
                int tz = z + g.off[0] - az;
                if (!fold_index(tz, g.T[0], g.wrap)) continue;
                for (int ay = 0; ay < g.A[1]; ++ay) {
                    int ty = y + g.off[1] - ay;
                    if (!fold_index(ty, g.T[1], g.wrap)) continue;
                    const T *hrow = h + ((long long)tz * g.T[1] + ty) * g.hsy;
                    const T *wrow = w + ((long long)az * g.A[1] + ay) * g.A[2];
                    for (int ax = 0; ax < g.A[2]; ++ax) {
                        int tx = x + g.off[2] - ax;
                        if (fold_index(tx, g.T[2], g.wrap)) acc += wrow[ax] * hrow[tx];
                    }
                }
            }
        }
        if (R) R[idx] = acc;
        if (V) {
            const double diff = (double)V[idx] - (double)acc;
            e_local += diff * diff;
        }
    }
    if (energy_partials) {
        const double s = block_sum_double<T>(e_local, red);
        if (threadIdx.x == 0) energy_partials[blockIdx.x] = s;
    }
}

// neg/pos[n,m,t] = sum_c sum_a W[m,c,a] * Xext[n,c,t-off+a], X = V / R     (tnmf/backends/NumPy.py:93-120)
// plus, when H is given, the fused multiplicative update (tnmf/TransformInvariantNMF.py:217-235,246-271).
// Only the activation indices [t_lo, t_lo + E[wax]) along axis `wax` (the first shift axis) are visited; E is T elsewhere.
template <typename T>
__global__ void __launch_bounds__(kGenericThreads)
generic_gradient_h_kernel(Geo g, const T *__restrict__ V, const T *__restrict__ R, const T *__restrict__ W,
                          T *__restrict__ neg_out, T *__restrict__ pos_out, T *__restrict__ H, T reg,
                          const T *__restrict__ G, T lambda, const T *__restrict__ Gsum, T lambda_cross,
                          int wax, int t_lo, int t_n) {
    const long long dvol = vol3(g.D), avol = vol3(g.A), tvol = vol3(g.T);
    const int E0 = wax == 0 ? t_n : g.T[0], E1 = wax == 1 ? t_n : g.T[1], E2 = wax == 2 ? t_n : g.T[2];
    const long long total = (long long)g.N * g.M * E0 * E1 * E2;
    for (long long w = (long long)blockIdx.x * blockDim.x + threadIdx.x; w < total;
         w += (long long)gridDim.x * blockDim.x) {
        long long r = w;
        const int tx = (int)(r % E2) + (wax == 2 ? t_lo : 0); r /= E2;
        const int ty = (int)(r % E1) + (wax == 1 ? t_lo : 0); r /= E1;
        const int tz = (int)(r % E0) + (wax == 0 ? t_lo : 0); r /= E0;
        const int m = (int)(r % g.M);
        const int n = (int)(r / g.M);
        const long long idx = (((long long)n * g.M + m) * g.T[0] + tz) * g.T[1] * g.T[2] + (long long)ty * g.T[2] + tx;
        T neg = 0, pos = 0;
        for (int c = 0; c < g.C; ++c) {
            const T *w = W + ((long long)m * g.C + c) * avol;
            const T *v = V + ((long long)n * g.C + c) * dvol;
            const T *rr = R + ((long long)n * g.C + c) * dvol;
            for (int az = 0; az < g.A[0]; ++az) {
                int z = tz - g.off[0] + az;
                if (!fold_index(z, g.D[0], g.wrap)) continue;
                for (int ay = 0; ay < g.A[1]; ++ay) {
                    int y = ty - g.off[1] + ay;
                    if (!fold_index(y, g.D[1], g.wrap)) continue;
                    const long long rowoff = ((long long)z * g.D[1] + y) * g.D[2];
                    const T *wrow = w + ((long long)az * g.A[1] + ay) * g.A[2];
                    for (int ax = 0; ax < g.A[2]; ++ax) {
                        int x = tx - g.off[2] + ax;
                        if (fold_index(x, g.D[2], g.wrap)) {
                            neg += wrow[ax] * v[rowoff + x];
                            pos += wrow[ax] * rr[rowoff + x];
                        }
                    }
                }
            }
        }
        if (H) {
            const long long tin = ((long long)tz * g.T[1] + ty) * g.T[2] + tx;
            T *hp = H + n * g.hsn + m * g.hsm + ((long long)tz * g.T[1] + ty) * g.hsy + tx;
            const T h = *hp;
            if (G) {
                const T gi = G[idx];
                if (lambda != (T)0) { T tmp = gi - h; tmp *= lambda; pos += tmp; }
                if (Gsum) { T tmp = -gi + Gsum[(long long)n * tvol + tin]; tmp *= lambda_cross; pos += tmp; }
            }
            pos += reg;
            T hn = h * neg;
            hn /= pos;
            *hp = hn;
        } else {
            neg_out[idx] = neg;
            pos_out[idx] = pos;
        }
    }
}

// neg/pos[m,c,a] = sum_n sum_d Hext[n,m,d+off-a] * X[n,c,d]               (tnmf/backends/NumPy.py:69-91)
// One block per output element; the reduction runs in double.  Activation indices outside [t_lo, t_hi) along axis `wax`
// (the first shift axis) do not contribute.
template <typename T>
__global__ void __launch_bounds__(kGenericThreads)
generic_gradient_w_kernel(Geo g, const T *__restrict__ V, const T *__restrict__ R, const T *__restrict__ H,
                          T *__restrict__ neg_out, T *__restrict__ pos_out, int wax, int t_lo, int t_hi) {
    __shared__ double red[32];
    const long long dvol = vol3(g.D);
    long long r = blockIdx.x;
    const int ax = (int)(r % g.A[2]); r /= g.A[2];
    const int ay = (int)(r % g.A[1]); r /= g.A[1];
    const int az = (int)(r % g.A[0]); r /= g.A[0];
    const int c = (int)(r % g.C);
    const int m = (int)(r / g.C);
    double neg = 0.0, pos = 0.0;
    const long long total = (long long)g.N * dvol;
    for (long long i = threadIdx.x; i < total; i += blockDim.x) {
        long long q = i;
        const int x = (int)(q % g.D[2]); q /= g.D[2];
        const int y = (int)(q % g.D[1]); q /= g.D[1];
        const int z = (int)(q % g.D[0]);
        const int n = (int)(q / g.D[0]);
        int tz = z + g.off[0] - az, ty = y + g.off[1] - ay, tx = x + g.off[2] - ax;
        if (!fold_index(tz, g.T[0], g.wrap) || !fold_index(ty, g.T[1], g.wrap) || !fold_index(tx, g.T[2], g.wrap))
            continue;
        const int tw = wax == 0 ? tz : wax == 1 ? ty : tx;
        if (tw < t_lo || tw >= t_hi) continue;
        const double h = (double)H[n * g.hsn + m * g.hsm + ((long long)tz * g.T[1] + ty) * g.hsy + tx];
        const long long xi = ((long long)n * g.C + c) * dvol + ((long long)z * g.D[1] + y) * g.D[2] + x;
        neg += h * (double)V[xi];
        pos += h * (double)R[xi];
    }
    neg = block_sum_double<T>(neg, red);
    __syncthreads();
    pos = block_sum_double<T>(pos, red);
    if (threadIdx.x == 0) {
        neg_out[blockIdx.x] = (T)neg;
        pos_out[blockIdx.x] = (T)pos;
    }
}

static inline int grid_for(long long total) {
    long long b = (total + kGenericThreads - 1) / kGenericThreads;
    if (b < 1) b = 1;
    return (int)(b > kGenericMaxBlocks ? kGenericMaxBlocks : b);
}

template <typename T>
int generic_reconstruct(const Geo &g, const T *W, const T *H, T *R, const T *V, double *energy_partials,
                        int *n_partials, cudaStream_t st) {
    const long long total = (long long)g.N * g.C * vol3(g.D);
    const int grid = grid_for(total);
    generic_reconstruct_kernel<T><<<grid, kGenericThreads, 0, st>>>(g, W, H, R, V, energy_partials);
    TNMF_CHECK_LAUNCH();
    if (n_partials) *n_partials = grid;
    return TNMF_OK;
}

template <typename T>
int generic_gradient_h(const Geo &g, const T *V, const T *R, const T *W, T *neg, T *pos, T *H, double reg,
                       const T *G, double lambda, const T *Gsum, double lambda_cross, cudaStream_t st, int t_lo,
                       int t_hi) {
    const int wax = 3 - g.ndim;
    if (t_hi < 0) { t_lo = 0; t_hi = g.T[wax]; }
    if (t_hi <= t_lo) return TNMF_OK;
    const long long total = (long long)g.N * g.M * (vol3(g.T) / g.T[wax]) * (t_hi - t_lo);
    generic_gradient_h_kernel<T><<<grid_for(total), kGenericThreads, 0, st>>>(
        g, V, R, W, neg, pos, H, (T)reg, G, (T)lambda, Gsum, (T)lambda_cross, wax, t_lo, t_hi - t_lo);
    TNMF_CHECK_LAUNCH();
    return TNMF_OK;
}

template <typename T>
int generic_gradient_w(const Geo &g, const T *V, const T *R, const T *H, T *neg, T *pos, cudaStream_t st, int t_lo,
                       int t_hi) {
    const long long outputs = (long long)g.M * g.C * vol3(g.A);
    if (outputs > 0x7fffffffLL) return TNMF_EUNSUPPORTED;
    const int wax = 3 - g.ndim;
    if (t_hi < 0) { t_lo = 0; t_hi = g.T[wax]; }
    generic_gradient_w_kernel<T><<<(int)outputs, kGenericThreads, 0, st>>>(g, V, R, H, neg, pos, wax, t_lo, t_hi);
    TNMF_CHECK_LAUNCH();
    return TNMF_OK;
}

#define INSTANTIATE(T)                                                                                          \
    template int generic_reconstruct<T>(const Geo &, const T *, const T *, T *, const T *, double *, int *,      \
                                        cudaStream_t);                                                          \
    template int generic_gradient_h<T>(const Geo &, const T *, const T *, const T *, T *, T *, T *, double,      \
                                       const T *, double, const T *, double, cudaStream_t, int, int);           \
    template int generic_gradient_w<T>(const Geo &, const T *, const T *, const T *, T *, T *, cudaStream_t, int, int);
INSTANTIATE(float)
INSTANTIATE(double)

}  // namespace tnmf
