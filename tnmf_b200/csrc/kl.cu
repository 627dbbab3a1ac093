// The elementwise pass of the Kullback-Leibler updates (DESIGN.md §3.11): Q = V / max(R, tau), Q = 0 where V = 0,
// written in place over R, and optionally the generalised KL divergence D(V||R) = sum V log(V / max(R, tau)) - V + R.
// With (Q, ones) in place of (V, R) the existing correlation kernels produce the KL gradients; this file is the only
// arithmetic the KL updates add.  HBM-bound: one read of V, one read and one write of R.
#include <cfloat>
#include "kl.cuh"

namespace tnmf {

namespace {

constexpr int kKlThreads = 256;
constexpr int kKlMaxBlocks = 2048;
constexpr int kKlPerThread = 4;         // elements one thread takes per sweep before the grid is capped

template <typename T> __device__ __forceinline__ T tiny();
template <> __device__ __forceinline__ float tiny<float>() { return FLT_MIN; }
template <> __device__ __forceinline__ double tiny<double>() { return DBL_MIN; }

// 16 bytes of consecutive elements: one 128-bit load / store
template <typename T> struct alignas(16) Pack { T x[16 / sizeof(T)]; };

// One element: returns Q and adds its divergence term, computed in double from the dtype inputs, to `acc`.  The IEEE
// division (no fast math in this library) rounds Q exactly like torch's `V / R.clamp(min=tau)` on the device.
template <typename T, bool DIV>
__device__ __forceinline__ T kl_element(T v, T r, double &acc) {
    const T rt = r < tiny<T>() ? tiny<T>() : r;
    if (DIV) {
        const double vd = v;
        acc += (v > T(0) ? vd * log(vd / (double)rt) : 0.0) - vd + (double)r;
    }
    return v > T(0) ? v / rt : T(0);
}

// Grid-stride over the elements (16-byte packs when both tensors are 16-byte aligned, then a scalar tail); with DIV each
// block writes the sum of its threads' terms, reduced in a fixed tree order, to partials[blockIdx.x].
template <typename T, bool DIV>
__global__ void __launch_bounds__(kKlThreads) kl_quotient_kernel(const T *__restrict__ V, T *__restrict__ R, long long n,
                                                                int packed, double *__restrict__ partials) {
    constexpr int L = 16 / sizeof(T);
    const long long stride = (long long)gridDim.x * kKlThreads;
    const long long tid = (long long)blockIdx.x * kKlThreads + threadIdx.x;
    double acc = 0.0;
    long long tail = 0;
    if (packed) {
        const long long np = n / L;
        for (long long i = tid; i < np; i += stride) {
            const Pack<T> v = reinterpret_cast<const Pack<T> *>(V)[i];
            Pack<T> r = reinterpret_cast<const Pack<T> *>(R)[i];
#pragma unroll
            for (int k = 0; k < L; ++k) r.x[k] = kl_element<T, DIV>(v.x[k], r.x[k], acc);
            reinterpret_cast<Pack<T> *>(R)[i] = r;
        }
        tail = np * L;
    }
    for (long long i = tail + tid; i < n; i += stride) R[i] = kl_element<T, DIV>(V[i], R[i], acc);
    if (!DIV) return;
    __shared__ double red[kKlThreads];
    red[threadIdx.x] = acc;
    __syncthreads();
    for (int o = kKlThreads / 2; o > 0; o >>= 1) {
        if (threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
        __syncthreads();
    }
    if (threadIdx.x == 0) partials[blockIdx.x] = red[0];
}

// D = sum of the per-block partials, in a fixed order
__global__ void __launch_bounds__(256) kl_finish_kernel(const double *__restrict__ partials, int n,
                                                       double *__restrict__ divergence) {
    __shared__ double red[256];
    double s = 0.0;
    for (int i = threadIdx.x; i < n; i += 256) s += partials[i];
    red[threadIdx.x] = s;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if (threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
        __syncthreads();
    }
    if (threadIdx.x == 0) *divergence = red[0];
}

bool aligned16(const void *p) { return (reinterpret_cast<unsigned long long>(p) & 15ull) == 0; }

}  // namespace

int kl_blocks(long long n) {
    const long long per_block = (long long)kKlThreads * kKlPerThread;
    const long long b = (n + per_block - 1) / per_block;
    return b < 1 ? 1 : b > kKlMaxBlocks ? kKlMaxBlocks : (int)b;
}

size_t kl_workspace_bytes(long long n) { return (sizeof(double) * (size_t)kl_blocks(n) + 255) & ~(size_t)255; }

template <typename T>
int kl_quotient(const T *V, T *R, long long n, double *divergence, void *workspace, cudaStream_t st) {
    const int blocks = kl_blocks(n);
    const int packed = aligned16(V) && aligned16(R);
    if (!divergence) {
        kl_quotient_kernel<T, false><<<blocks, kKlThreads, 0, st>>>(V, R, n, packed, nullptr);
        TNMF_CHECK_LAUNCH();
        return TNMF_OK;
    }
    double *partials = (double *)workspace;
    kl_quotient_kernel<T, true><<<blocks, kKlThreads, 0, st>>>(V, R, n, packed, partials);
    TNMF_CHECK_LAUNCH();
    kl_finish_kernel<<<1, 256, 0, st>>>(partials, blocks, divergence);
    TNMF_CHECK_LAUNCH();
    return TNMF_OK;
}
template int kl_quotient<float>(const float *, float *, long long, double *, void *, cudaStream_t);
template int kl_quotient<double>(const double *, double *, long long, double *, void *, cudaStream_t);

}  // namespace tnmf
