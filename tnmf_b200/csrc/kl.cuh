// The Kullback-Leibler pass (kl.cu): the quotient Q = V / max(R, tau) written over R, and optionally the divergence.
#pragma once
#include "common.cuh"

namespace tnmf {

// per-block partials of the divergence: the grid depends on the element count only
int kl_blocks(long long n);
size_t kl_workspace_bytes(long long n);
template <typename T>
int kl_quotient(const T *V, T *R, long long n, double *divergence, void *workspace, cudaStream_t st);

}  // namespace tnmf
