// extern "C" surface of libtnmf_b200.so: argument validation, geometry set-up, kernel choice and dispatch.
// See include/tnmf_b200.h for the contract of every entry point and the reference interface it replaces.
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include "common.cuh"

using namespace tnmf;

static bool aligned16(const void *p) { return (reinterpret_cast<unsigned long long>(p) & 15ull) == 0; }

namespace {

// A batch of single-channel 1-D signals IS one 2-D image: row n = signal n, atoms one row high (A_y = 1, so rows never
// mix).  V[n,0,x], R[n,0,x] and W[m,0,a] are already laid out that way; H[n,m,t] becomes the image's activation with
// the sample stride as its row stride.  The 2-D kernel families (TMA staging, persistent CTAs) then serve the 1-D
// problems as well - cfg4 (2048 x 4096, 64 atoms x 128): 28.1 -> 23.1 ms per iteration on B200.  Offsets inside one
// "image" are 32-bit in the tiled kernels, hence the size guard; tnmf_problem.flags: TNMF_FLAG_NO_ROWS_VIEW keeps the 1-D
// kernels, TNMF_FLAG_ROWS_VIEW_ALWAYS takes the view whatever the batch size (default: from 2^20 signal elements on).
void rows_view(const tnmf_problem *p, Geo &g) {
    if (p->ndim != 1 || g.C != 1 || g.wrap || p->dtype != TNMF_F32 || g.N < 2) return;
    if ((long long)g.N * g.D[2] >= (1ll << 30) || (long long)g.N * g.T[2] >= (1ll << 30)) return;
    if (p->flags & TNMF_FLAG_NO_ROWS_VIEW) return;
    // small batches do not fill the persistent 2-D kernels (cfg1, 100 x 1000: 0.079 against 0.060 ms per iteration)
    if (!(p->flags & TNMF_FLAG_ROWS_VIEW_ALWAYS) && (long long)g.N * g.D[2] < (1ll << 20)) return;
    g.D[1] = g.N; g.T[1] = g.N; g.A[1] = 1; g.off[1] = 0;
    g.hsy = g.hsn;
    g.hsn = g.hsn * g.N;
    g.N = 1;
    g.ndim = 2;
}

int make_geo(const tnmf_problem *p, Geo &g, bool allow_rows_view = true) {
    if (!p) return TNMF_EINVAL;
    if (p->ndim < 1 || p->ndim > TNMF_MAX_SHIFT_DIMS) return TNMF_EUNSUPPORTED;
    if (p->dtype != TNMF_F32 && p->dtype != TNMF_F64) return TNMF_EUNSUPPORTED;
    if (p->mode != TNMF_VALID && p->mode != TNMF_FULL && p->mode != TNMF_CIRCULAR) return TNMF_EINVAL;
    if (p->n_samples < 0 || p->n_channels < 1 || p->n_atoms < 1 || p->reserved != 0) return TNMF_EINVAL;
    g.N = p->n_samples; g.C = p->n_channels; g.M = p->n_atoms; g.ndim = p->ndim;
    g.wrap = p->mode == TNMF_CIRCULAR;
    g.flags = p->flags;
    const int lead = 3 - p->ndim;
    for (int i = 0; i < 3; ++i) { g.D[i] = 1; g.A[i] = 1; g.T[i] = 1; g.off[i] = 0; }
    for (int i = 0; i < p->ndim; ++i) {
        const int d = p->sample_shape[i], a = p->atom_shape[i];
        if (d < 1 || a < 1) return TNMF_EINVAL;
        int t;
        if (p->mode == TNMF_VALID) t = d + a - 1;
        else if (p->mode == TNMF_FULL) t = d - a + 1;
        else t = d;
        if (t < 1) return TNMF_EINVAL;
        g.D[lead + i] = d; g.A[lead + i] = a; g.T[lead + i] = t;
        g.off[lead + i] = p->mode == TNMF_VALID ? a - 1 : 0;
    }
    if (p->h_pitch != 0 && p->h_pitch < g.T[2]) return TNMF_EINVAL;
    g.hsy = p->h_pitch ? p->h_pitch : g.T[2];
    const long long tvol = (long long)g.T[0] * g.T[1] * g.hsy;
    g.hsm = p->h_stride_m ? p->h_stride_m : tvol;
    g.hsn = p->h_stride_n ? p->h_stride_n : tvol * g.M;
    if (allow_rows_view) rows_view(p, g);
    return TNMF_OK;
}

// The tensor-core H update pads the contraction C*A_x to a multiple of 8 and the atoms to a multiple of 16; 'auto'
// takes it when at least half of every MMA is useful work and the problem fills the 128-column tiles
// (TNMF_FLAG_NO_TC_HUPD keeps 'auto' on the FP32 kernels).
bool tc_worthwhile(const Geo &g) {
    if (g.flags & TNMF_FLAG_NO_TC_HUPD) return false;
    const int k = g.C * g.A[2], kp = (k + 7) / 8 * 8, mp = (g.M + 15) / 16 * 16;
    const double useful = ((double)k / kp) * ((double)g.M / mp);
    return useful >= 0.5 && (long long)g.N * g.T[2] >= 128 && g.A[1] >= 3;
}

// The tensor-core reconstruction has N = roundup(A_y * C, 16) <= 64: every MMA sits on the per-instruction floor, so it
// pays when many (atom row, channel) pairs share one MMA and the atoms fill the K steps (TNMF_FLAG_NO_TC_RECON keeps FP32).
bool tc_recon_worthwhile(const Geo &g) {
    if (g.flags & TNMF_FLAG_NO_TC_RECON) return false;
    const int km = (g.M + 7) / 8 * 8;
    return g.A[1] * g.C >= 24 && (double)g.M / km >= 0.75 && (long long)g.N * g.D[2] >= 128;
}

// The tensor-core W gradient stacks the expanded V and R rows (of two consecutive source rows when the atom is narrow)
// into the 128 MMA lanes: 2 * S * roundup(C*A_x, 8) of them carry taps.  'auto' takes it when that is at least half of
// the tile (TNMF_FLAG_NO_TC_GRADW keeps the FP32 kernel).
bool tc_gradw_worthwhile(const Geo &g) {
    if (g.flags & TNMF_FLAG_NO_TC_GRADW) return false;
    const int kp = (g.C * g.A[2] + 7) / 8 * 8, mp = (g.M + 15) / 16 * 16;
    const int stack = (4 * kp <= 128 && 16 * (g.A[1] + 1) <= 256) ? 2 : 1;
    // atoms higher than 15 rows run in row chunks that expand V and R once per chunk: measured no faster than the FP32
    // kernel (cfg5: 11.2 against 11.0 ms), so 'auto' leaves them there; kernel_path='tc' still takes the chunked form
    return 2 * stack * kp >= 64 && g.C * g.A[2] * 2 >= kp && (double)g.M / mp >= 0.5 && (long long)g.N * g.T[2] >= 64 &&
           g.A[1] >= 3 && g.A[1] <= 15;
}

// The W gradient for narrow atoms (tc_gradw_ns.cu: C * A_x <= 16; hi / lo halves, two source rows and both tensors stacked
// in the 128 MMA lanes, two MMAs per product): 'auto' takes it when at least half of the lanes carry taps.
bool tc_gradw_ns_worthwhile(const Geo &g) {
    if (g.flags & TNMF_FLAG_NO_TC_GRADW) return false;
    const int mp = (g.M + 7) / 8 * 8;
    return 8 * g.C * g.A[2] >= 64 && (double)g.M / mp >= 0.5 && (long long)g.N * g.T[2] >= 64 && g.A[1] >= 3;
}

// The reconstructions with a tensor-memory ring - of activation rows (tc_recon_ts.cu: N = roundup(C * A_x, 16)) or, for
// what that kernel cannot hold (one channel, many atoms: cfg3), of output-row accumulators (tc_recon_os.cu: one MMA of
// N = A_y * roundup(C * A_x, 16) per source row and K step).  K = atoms padded to 8, and 128 - (A_x - 1) of the 128 MMA
// lanes produce outputs; 'auto' takes them when at least half of every MMA is useful work.
bool tc_recon_tmem_worthwhile(const Geo &g) {
    if (g.flags & TNMF_FLAG_NO_TC_RECON) return false;
    const int nu = g.C * g.A[2], np = (nu + 15) / 16 * 16, km = (g.M + 7) / 8 * 8;
    const double useful = ((double)nu / np) * ((double)g.M / km) * (double)(128 - (g.A[2] - 1)) / 128.0;
    // (one-row atoms - 1-D batches run as an image of signal rows - would contract over the atoms only: MMAs too small)
    return useful >= 0.5 && (long long)g.N * g.D[2] >= 128 && g.A[1] >= 3;
}

// Every hot kernel an operation can run on.  The FP32 and generic families have one kernel per operation and share the
// values of their TNMF_PATH_*; every other value is a tensor-core kernel (family TNMF_PATH_TC).
enum Kernel {
    K_NONE = -1,
    K_GENERIC = TNMF_PATH_GENERIC, K_TILED = TNMF_PATH_TILED, K_TMA = TNMF_PATH_TMA,
    K_RECON_TS = TNMF_PATH_TC, K_RECON_OS, K_RECON_TC, K_HUPD_TS, K_HUPD_TC, K_GRADW_TS, K_GRADW_NS, K_GRADW_TC,
    K_RECON_OS3, K_HUPD_TS3, K_GRADW_NS3,                      // the 3-D plane mode of recon_os, hupd_ts and gradw_ns
};

int kernel_family(int k) { return k < TNMF_PATH_TC ? k : TNMF_PATH_TC; }

// The kernel that serves operation `op`, or K_NONE with *err set when a forced family cannot serve the problem.  'auto'
// takes a tensor-core kernel where it plans and is worthwhile, the tensor-memory operand kernels before the round-1 ones;
// else the TMA kernels where eligible, else the cp.async tiled ones, else the generic ones.  Forced 'tc' takes a
// tensor-core kernel wherever one plans and otherwise goes on like 'auto'.
int plan_kernel(const tnmf_problem *p, const Geo &g, int op, int *err) {
    *err = TNMF_OK;
    if (p->path == TNMF_PATH_GENERIC) return K_GENERIC;
    const int dt = p->dtype;
    const bool forced = p->path == TNMF_PATH_TC, autop = p->path == TNMF_PATH_AUTO;
    const bool tmem = !(g.flags & TNMF_FLAG_NO_TMEM_OPERAND);
    if (plane_problem(g)) {
        // 3-D problems run on the plane mode of three tensor-memory kernels (DESIGN.md §3.10), float32 'valid' only.
        // Their alternative is the generic kernel, not the FP32 tiled / TMA ones (2-D only), so 'auto' takes them
        // wherever they plan and at least half of every 16-atom block is real atoms (a few atoms in a large padded MMA
        // lose to nothing).  The TNMF_FLAG_NO_TC_* flags keep 'auto' on the generic kernels, TNMF_FLAG_NO_TMEM_OPERAND
        // keeps every path there.
        static const int no_tc[3] = {TNMF_FLAG_NO_TC_RECON, TNMF_FLAG_NO_TC_HUPD, TNMF_FLAG_NO_TC_GRADW};
        if (tmem && (forced || (autop && !(g.flags & no_tc[op]) && (double)g.M / ((g.M + 15) / 16 * 16) >= 0.5))) {
            if (op == TNMF_OP_RECONSTRUCT && tc_recon_os_supported(g, dt)) return K_RECON_OS3;
            if (op == TNMF_OP_GRADIENT_H && tc_hupd_ts_supported(g, dt)) return K_HUPD_TS3;
            if (op == TNMF_OP_GRADIENT_W && tc_gradw_ns_supported(g, dt)) return K_GRADW_NS3;
        }
        if (p->path == TNMF_PATH_TMA || p->path == TNMF_PATH_TILED) { *err = TNMF_EUNSUPPORTED; return K_NONE; }
        return K_GENERIC;                                           // forced 'tc': tensor cores where a kernel plans
    }
    bool tma_ok = false;
    if (op == TNMF_OP_RECONSTRUCT) {
        const bool tmem_want = forced || (autop && tc_recon_tmem_worthwhile(g));
        if (tmem && tmem_want && tc_recon_ts_supported(g, dt)) return K_RECON_TS;
        if (tmem && tmem_want && tc_recon_os_supported(g, dt)) return K_RECON_OS;
        if ((forced || (autop && tc_recon_worthwhile(g))) && tc_recon_supported(g, dt)) return K_RECON_TC;
        tma_ok = tma_recon_supported(g, dt);
    } else if (op == TNMF_OP_GRADIENT_H) {
        if (forced || (autop && tc_worthwhile(g))) {
            if (tmem && tc_hupd_ts_supported(g, dt)) return K_HUPD_TS;
            if (tc_hupd_supported(g, dt)) return K_HUPD_TC;
        }
        tma_ok = tma_hupd_supported(g, dt);
    } else {
        if (tmem && (forced || (autop && tc_gradw_ns_worthwhile(g))) && tc_gradw_ns_supported(g, dt)) return K_GRADW_NS;
        if (forced || (autop && tc_gradw_worthwhile(g))) {
            if (tmem && tc_gradw_ts_supported(g, dt)) return K_GRADW_TS;
            if (tc_gradw_supported(g, dt)) return K_GRADW_TC;
        }
        tma_ok = tma_gradw_supported(g, dt);
    }
    if (tma_ok && (autop || forced || p->path == TNMF_PATH_TMA)) return K_TMA;
    if (p->path == TNMF_PATH_TMA) { *err = TNMF_EUNSUPPORTED; return K_NONE; }
    if (tiled_supported(g, dt)) return K_TILED;
    if (p->path == TNMF_PATH_TILED) { *err = TNMF_EUNSUPPORTED; return K_NONE; }
    return K_GENERIC;
}

// The TMA kernels need 16-byte aligned operands (`aligned`: those the caller's kernel reads) and a workspace for the
// pre-arranged atoms: without them a forced 'tma' is an error, and the other paths fall back to the tiled kernels, else
// the generic ones.
int tma_fallback(const tnmf_problem *p, const Geo &g, int &k, bool aligned, bool workspace) {
    if (k != K_TMA || (aligned && workspace)) return TNMF_OK;
    if (p->path == TNMF_PATH_TMA) return workspace ? TNMF_EUNSUPPORTED : TNMF_EWORKSPACE;
    k = tiled_supported(g, p->dtype) ? K_TILED : K_GENERIC;
    return TNMF_OK;
}

size_t align256(size_t b) { return (b + 255) & ~(size_t)255; }

size_t energy_partials_bytes(const Geo &g) {
    return align256(sizeof(double) * (size_t)generic_energy_partial_capacity(g));
}

// the 3-D tensor-core reconstruction accumulates R over its per-plane launches: without a caller's R buffer it needs
// R-sized scratch (behind the energy partials in the workspace)
size_t r_scratch_bytes(const Geo &g) { return align256(sizeof(float) * (size_t)g.N * g.C * (size_t)vol3(g.D)); }

}  // namespace

extern "C" {

int tnmf_abi_version(void) { return TNMF_ABI_VERSION; }

const char *tnmf_status_string(int status) {
    static thread_local char buf[160];
    switch (status) {
        case TNMF_OK: return "ok";
        case TNMF_EINVAL: return "invalid argument";
        case TNMF_EUNSUPPORTED: return "unsupported problem (no kernel, and there is no CPU fallback)";
        case TNMF_EWORKSPACE: return "workspace too small";
        default: break;
    }
    if (status >= TNMF_ECUDA) {
        snprintf(buf, sizeof(buf), "CUDA error %d: %s", status - TNMF_ECUDA,
                 cudaGetErrorString((cudaError_t)(status - TNMF_ECUDA)));
        return buf;
    }
    return "unknown status";
}

int tnmf_transform_shape(const tnmf_problem *p, int32_t *t_shape) {
    Geo g;
    int s = make_geo(p, g);
    if (s) return s;
    if (!t_shape) return TNMF_EINVAL;
    for (int i = 0; i < p->ndim; ++i) t_shape[i] = g.T[3 - p->ndim + i];
    return TNMF_OK;
}

static size_t workspace_bytes_of(const Geo &g, int dtype) {
    size_t bytes = energy_partials_bytes(g);
    if (tiled_supported(g, dtype)) {
        const size_t t = align256(tiled_workspace_bytes(g));
        if (t > bytes) bytes = t;
    }
    const size_t t = tma_workspace_bytes(g, dtype);
    if (t > bytes) bytes = t;
    if (tc_gradw_supported(g, dtype)) {
        const size_t w = align256(tc_gradw_workspace_bytes(g));
        if (w > bytes) bytes = w;
    }
    if (tc_gradw_ts_supported(g, dtype)) {
        const size_t w = align256(tc_gradw_ts_workspace_bytes(g));
        if (w > bytes) bytes = w;
    }
    if (tc_gradw_ns_supported(g, dtype)) {
        const size_t w = align256(tc_gradw_ns_workspace_bytes(g));
        if (w > bytes) bytes = w;
    }
    if (tc_recon_os_supported(g, dtype) && plane_problem(g)) {
        const size_t w = energy_partials_bytes(g) + r_scratch_bytes(g);
        if (w > bytes) bytes = w;
    }
    return bytes;
}

size_t tnmf_workspace_bytes(const tnmf_problem *p) {
    Geo g, plain;
    if (make_geo(p, g) || make_geo(p, plain, false)) return 0;
    const size_t a = workspace_bytes_of(g, p->dtype), b = workspace_bytes_of(plain, p->dtype);
    return a > b ? a : b;
}

int tnmf_uses_tiled_path(const tnmf_problem *p) {
    Geo g;
    if (make_geo(p, g)) return 0;
    int err;
    const int k = plan_kernel(p, g, TNMF_OP_GRADIENT_H, &err);
    return k != K_NONE && k != K_GENERIC;
}

int tnmf_kernel_family(const tnmf_problem *p, int op) {
    Geo g;
    if (make_geo(p, g)) return -1;
    if (op < TNMF_OP_RECONSTRUCT || op > TNMF_OP_GRADIENT_W) return -1;
    int err;
    return kernel_family(plan_kernel(p, g, op, &err));
}

const char *tnmf_kernel_name(const tnmf_problem *p, int op) {
    Geo g;
    if (make_geo(p, g) || op < TNMF_OP_RECONSTRUCT || op > TNMF_OP_GRADIENT_W) return "none";
    int err;
    static const char *const fp32[3][3] = {   // [kernel - K_GENERIC][op]
        {"generic_reconstruct_kernel", "generic_gradient_h_kernel", "generic_gradient_w_kernel"},
        {"tiled::recon_kernel", "tiled::hupd_kernel", "tiled::gradw_kernel"},
        {"recon_tma_kernel", "hupd_tma_kernel", "gradw_tma_kernel"}};
    const int k = plan_kernel(p, g, op, &err);
    switch (k) {
        case K_GENERIC: case K_TILED: case K_TMA: return fp32[k - K_GENERIC][op];
        case K_RECON_TS: return "recon_ts_kernel";
        case K_RECON_OS: return "recon_os_kernel";
        case K_RECON_TC: return "recon_tc_kernel";
        case K_HUPD_TS: return "hupd_ts_kernel";
        case K_HUPD_TC: return "hupd_tc_kernel";
        case K_GRADW_TS: return "gradw_ts_kernel";
        case K_GRADW_NS: return "gradw_ns_kernel";
        case K_GRADW_TC: return "gradw_tc_kernel";
        case K_RECON_OS3: return "recon_os3_kernel";
        case K_HUPD_TS3: return "hupd_ts3_kernel";
        case K_GRADW_NS3: return "gradw_ns3_kernel";
        default: return "none";
    }
}

int tnmf_launch_count(const tnmf_problem *p, int op) {
    Geo g;
    if (make_geo(p, g)) return -1;
    if (op < TNMF_OP_RECONSTRUCT || op > TNMF_OP_GRADIENT_W) return -1;
    int err;
    switch (plan_kernel(p, g, op, &err)) {
        case K_GENERIC: case K_TILED: return op == TNMF_OP_GRADIENT_W ? 2 : 1;     // + the finishing reduction
        case K_TMA: return 2;                                   // + the atom pre-arrangement / the finishing reduction
        case K_RECON_TS: case K_RECON_TC: return 1;
        case K_RECON_OS: case K_RECON_OS3: return tc_recon_os_launches(g);
        case K_HUPD_TS: case K_HUPD_TS3: return tc_hupd_ts_launches(g);
        case K_HUPD_TC: return tc_hupd_launches(g);
        case K_GRADW_TS: return tc_gradw_ts_launches(g);
        case K_GRADW_NS: case K_GRADW_NS3: return tc_gradw_ns_launches(g);
        case K_GRADW_TC: return tc_gradw_launches(g);
        default: return -1;
    }
}

// The reconstruction behind tnmf_reconstruct (V, partials: null) and tnmf_reconstruct_energy (the TMA kernels keep their
// energy partials at their own place in the workspace)
static int reconstruct_dispatch(const tnmf_problem *p, const Geo &g, int k, const void *W, const void *H, void *R,
                                const void *V, double *&partials, int *n_partials, void *workspace,
                                size_t workspace_bytes, cudaStream_t st) {
    switch (k) {
        case K_RECON_TS:
            return tc_reconstruct_ts(g, (const float *)W, (const float *)H, (float *)R, (const float *)V, partials,
                                     n_partials, st);
        case K_RECON_OS3:                       // (an energy without a caller's R accumulates in workspace scratch)
            if (!R) R = (char *)workspace + energy_partials_bytes(g);
            [[fallthrough]];
        case K_RECON_OS:
            return tc_reconstruct_os(g, (const float *)W, (const float *)H, (float *)R, (const float *)V, partials,
                                     n_partials, st);
        case K_RECON_TC:
            return tc_reconstruct(g, (const float *)W, (const float *)H, (float *)R, (const float *)V, partials,
                                  n_partials, st);
        case K_TMA:
            if (V) partials = tma_energy_partials(g, workspace);
            return tma_reconstruct(g, (const float *)W, (const float *)H, (float *)R, (const float *)V, partials,
                                   n_partials, workspace, workspace_bytes, st);
        case K_TILED:
            return tiled_reconstruct(g, (const float *)W, (const float *)H, (float *)R, (const float *)V, partials,
                                     n_partials, st);
        case K_GENERIC: break;
        default: return TNMF_EUNSUPPORTED;
    }
    if (p->dtype == TNMF_F32)
        return generic_reconstruct<float>(g, (const float *)W, (const float *)H, (float *)R, (const float *)V, partials,
                                          n_partials, st);
    return generic_reconstruct<double>(g, (const double *)W, (const double *)H, (double *)R, (const double *)V,
                                       partials, n_partials, st);
}

int tnmf_reconstruct(const tnmf_problem *p, const void *W, const void *H, void *R, void *workspace,
                     size_t workspace_bytes, void *stream) {
    Geo g;
    int s = make_geo(p, g);
    if (s) return s;
    if (!W || !H || !R) return TNMF_EINVAL;
    if (g.N == 0) return TNMF_OK;
    int k = plan_kernel(p, g, TNMF_OP_RECONSTRUCT, &s);
    if (s || (s = tma_fallback(p, g, k, aligned16(H), workspace))) return s;
    double *partials = nullptr;
    return reconstruct_dispatch(p, g, k, W, H, R, nullptr, partials, nullptr, workspace, workspace_bytes,
                                (cudaStream_t)stream);
}

int tnmf_reconstruct_energy(const tnmf_problem *p, const void *V, const void *W, const void *H, void *R,
                            double *energy, void *workspace, size_t workspace_bytes, void *stream) {
    Geo g;
    int s = make_geo(p, g);
    if (s) return s;
    if (!V || !W || !H || !energy || !workspace) return TNMF_EINVAL;
    if (workspace_bytes < tnmf_workspace_bytes(p)) return TNMF_EWORKSPACE;
    cudaStream_t st = (cudaStream_t)stream;
    double *partials = (double *)workspace;
    int n_partials = 0;
    if (g.N == 0) {
        cudaError_t e = cudaMemsetAsync(energy, 0, sizeof(double), st);
        return status_from_cuda(e);
    }
    int k = plan_kernel(p, g, TNMF_OP_RECONSTRUCT, &s);
    if (s || (s = tma_fallback(p, g, k, aligned16(H), workspace))) return s;
    s = reconstruct_dispatch(p, g, k, W, H, R, V, partials, &n_partials, workspace, workspace_bytes, st);
    if (s) return s;
    return finish_energy(partials, n_partials, energy, st);
}

static int gradient_h_dispatch(const tnmf_problem *p, const void *V, const void *R, const void *W, void *neg,
                               void *pos, void *H, double reg, const void *G, double lambda, const void *Gsum,
                               double lambda_cross, void *workspace, size_t workspace_bytes, void *stream) {
    Geo g;
    // the rows view re-strides H only: dense neg / pos outputs and dense G / Gsum inputs are in the caller's
    // [n][m][t] order, so the unfused gradient and the inhibition epilogue keep the 1-D geometry
    int s = make_geo(p, g, !neg && !pos && !G && !Gsum);
    if (s) return s;
    if (!V || !R || !W) return TNMF_EINVAL;
    if (g.N == 0) return TNMF_OK;
    cudaStream_t st = (cudaStream_t)stream;
    int k = plan_kernel(p, g, TNMF_OP_GRADIENT_H, &s);
    if (s || (s = tma_fallback(p, g, k, aligned16(V) && aligned16(R), workspace))) return s;
    switch (k) {
        case K_HUPD_TS: case K_HUPD_TS3:
            return tc_gradient_h_ts(g, (const float *)V, (const float *)R, (const float *)W, (float *)neg, (float *)pos,
                                    (float *)H, reg, (const float *)G, lambda, (const float *)Gsum, lambda_cross, st);
        case K_HUPD_TC:
            return tc_gradient_h(g, (const float *)V, (const float *)R, (const float *)W, (float *)neg, (float *)pos,
                                 (float *)H, reg, (const float *)G, lambda, (const float *)Gsum, lambda_cross, st);
        case K_TMA:
            return tma_gradient_h(g, (const float *)V, (const float *)R, (const float *)W, (float *)neg, (float *)pos,
                                  (float *)H, reg, (const float *)G, lambda, (const float *)Gsum, lambda_cross,
                                  workspace, workspace_bytes, st);
        case K_TILED:
            return tiled_gradient_h(g, (const float *)V, (const float *)R, (const float *)W, (float *)neg, (float *)pos,
                                    (float *)H, reg, (const float *)G, lambda, (const float *)Gsum, lambda_cross, st);
        case K_GENERIC: break;
        default: return TNMF_EUNSUPPORTED;
    }
    if (p->dtype == TNMF_F32)
        return generic_gradient_h<float>(g, (const float *)V, (const float *)R, (const float *)W, (float *)neg,
                                         (float *)pos, (float *)H, reg, (const float *)G, lambda,
                                         (const float *)Gsum, lambda_cross, st);
    return generic_gradient_h<double>(g, (const double *)V, (const double *)R, (const double *)W, (double *)neg,
                                      (double *)pos, (double *)H, reg, (const double *)G, lambda,
                                      (const double *)Gsum, lambda_cross, st);
}

int tnmf_gradient_h(const tnmf_problem *p, const void *V, const void *R, const void *W, void *neg, void *pos,
                    void *workspace, size_t workspace_bytes, void *stream) {
    if (!neg || !pos) return TNMF_EINVAL;
    return gradient_h_dispatch(p, V, R, W, neg, pos, nullptr, 0.0, nullptr, 0.0, nullptr, 0.0, workspace,
                               workspace_bytes, stream);
}

int tnmf_update_h(const tnmf_problem *p, const void *V, const void *R, const void *W, void *H, double reg,
                  const void *G, double lambda, const void *Gsum, double lambda_cross, void *workspace,
                  size_t workspace_bytes, void *stream) {
    if (!H) return TNMF_EINVAL;
    if (lambda_cross != 0.0 && !Gsum) return TNMF_EINVAL;
    if (lambda_cross == 0.0) Gsum = nullptr;
    if (lambda == 0.0 && !Gsum) G = nullptr;
    if ((lambda != 0.0 || Gsum) && !G) return TNMF_EINVAL;
    return gradient_h_dispatch(p, V, R, W, nullptr, nullptr, H, reg, G, lambda, Gsum, lambda_cross, workspace,
                               workspace_bytes, stream);
}

int tnmf_gradient_w(const tnmf_problem *p, const void *V, const void *R, const void *H, void *neg, void *pos,
                    void *workspace, size_t workspace_bytes, void *stream) {
    Geo g;
    int s = make_geo(p, g);
    if (s) return s;
    if (!V || !R || !H || !neg || !pos) return TNMF_EINVAL;
    cudaStream_t st = (cudaStream_t)stream;
    const size_t esz = p->dtype == TNMF_F32 ? 4 : 8;
    const size_t count = (size_t)g.M * g.C * (size_t)vol3(g.A);
    if (g.N == 0) {
        cudaError_t e = cudaMemsetAsync(neg, 0, count * esz, st);
        if (e == cudaSuccess) e = cudaMemsetAsync(pos, 0, count * esz, st);
        return status_from_cuda(e);
    }
    int k = plan_kernel(p, g, TNMF_OP_GRADIENT_W, &s);
    // every W gradient but the generic one needs the workspace, so a missing one is an error rather than a fallback
    if (s || (s = tma_fallback(p, g, k, aligned16(V) && aligned16(R) && aligned16(H), true))) return s;
    if (k != K_GENERIC && (!workspace || workspace_bytes < tnmf_workspace_bytes(p))) return TNMF_EWORKSPACE;
    switch (k) {
        case K_GRADW_NS: case K_GRADW_NS3:
            return tc_gradient_w_ns(g, (const float *)V, (const float *)R, (const float *)H, (float *)neg, (float *)pos,
                                    workspace, workspace_bytes, st);
        case K_GRADW_TS:
            return tc_gradient_w_ts(g, (const float *)V, (const float *)R, (const float *)H, (float *)neg, (float *)pos,
                                    workspace, workspace_bytes, st);
        case K_GRADW_TC:
            return tc_gradient_w(g, (const float *)V, (const float *)R, (const float *)H, (float *)neg, (float *)pos,
                                 workspace, workspace_bytes, st);
        case K_TMA:
            return tma_gradient_w(g, (const float *)V, (const float *)R, (const float *)H, (float *)neg, (float *)pos,
                                  workspace, workspace_bytes, st);
        case K_TILED:
            return tiled_gradient_w(g, (const float *)V, (const float *)R, (const float *)H, (float *)neg, (float *)pos,
                                    workspace, workspace_bytes, st);
        case K_GENERIC: break;
        default: return TNMF_EUNSUPPORTED;
    }
    if (p->dtype == TNMF_F32)
        return generic_gradient_w<float>(g, (const float *)V, (const float *)R, (const float *)H, (float *)neg,
                                         (float *)pos, st);
    return generic_gradient_w<double>(g, (const double *)V, (const double *)R, (const double *)H, (double *)neg,
                                      (double *)pos, st);
}

// The plane-window entry points: the kernels that serve them are the plane mode of the tensor-memory kernels (3-D float32
// 'valid') and the generic kernels; every other family has no window and the call is unsupported.  The window is on the
// first shift axis of the problem as the caller describes it (no rows view).
static int window_kernel(const tnmf_problem *p, Geo &g, int op, int t_lo, int t_hi, int *k) {
    int s = make_geo(p, g, false);
    if (s) return s;
    const int wax = 3 - p->ndim;
    if (t_lo < 0 || t_hi < t_lo || t_hi > g.T[wax]) return TNMF_EINVAL;
    *k = plan_kernel(p, g, op, &s);
    if (s) return s;
    return *k == K_GENERIC || *k == K_HUPD_TS3 || *k == K_GRADW_NS3 ? TNMF_OK : TNMF_EUNSUPPORTED;
}

int tnmf_update_h_planes(const tnmf_problem *p, const void *V, const void *R, const void *W, void *H, double reg,
                         const void *G, double lambda, const void *Gsum, double lambda_cross, int32_t t_lo, int32_t t_hi,
                         void *workspace, size_t workspace_bytes, void *stream) {
    (void)workspace; (void)workspace_bytes;
    if (!H || !V || !R || !W) return TNMF_EINVAL;
    if (lambda_cross != 0.0 && !Gsum) return TNMF_EINVAL;
    if (lambda_cross == 0.0) Gsum = nullptr;
    if (lambda == 0.0 && !Gsum) G = nullptr;
    if ((lambda != 0.0 || Gsum) && !G) return TNMF_EINVAL;
    Geo g;
    int k;
    int s = window_kernel(p, g, TNMF_OP_GRADIENT_H, t_lo, t_hi, &k);
    if (s) return s;
    if (g.N == 0 || t_lo == t_hi) return TNMF_OK;
    cudaStream_t st = (cudaStream_t)stream;
    if (k == K_HUPD_TS3)
        return tc_gradient_h_ts(g, (const float *)V, (const float *)R, (const float *)W, nullptr, nullptr, (float *)H, reg,
                                (const float *)G, lambda, (const float *)Gsum, lambda_cross, st, t_lo, t_hi);
    if (p->dtype == TNMF_F32)
        return generic_gradient_h<float>(g, (const float *)V, (const float *)R, (const float *)W, nullptr, nullptr,
                                         (float *)H, reg, (const float *)G, lambda, (const float *)Gsum, lambda_cross,
                                         st, t_lo, t_hi);
    return generic_gradient_h<double>(g, (const double *)V, (const double *)R, (const double *)W, nullptr, nullptr,
                                      (double *)H, reg, (const double *)G, lambda, (const double *)Gsum, lambda_cross,
                                      st, t_lo, t_hi);
}

int tnmf_gradient_w_planes(const tnmf_problem *p, const void *V, const void *R, const void *H, void *neg, void *pos,
                           int32_t t_lo, int32_t t_hi, void *workspace, size_t workspace_bytes, void *stream) {
    if (!V || !R || !H || !neg || !pos) return TNMF_EINVAL;
    Geo g;
    int k;
    int s = window_kernel(p, g, TNMF_OP_GRADIENT_W, t_lo, t_hi, &k);
    if (s) return s;
    cudaStream_t st = (cudaStream_t)stream;
    if (g.N == 0) {
        const size_t bytes = (size_t)g.M * g.C * (size_t)vol3(g.A) * (p->dtype == TNMF_F32 ? 4 : 8);
        cudaError_t e = cudaMemsetAsync(neg, 0, bytes, st);
        if (e == cudaSuccess) e = cudaMemsetAsync(pos, 0, bytes, st);
        return status_from_cuda(e);
    }
    if (k == K_GRADW_NS3) {
        if (!workspace || workspace_bytes < tnmf_workspace_bytes(p)) return TNMF_EWORKSPACE;
        return tc_gradient_w_ns(g, (const float *)V, (const float *)R, (const float *)H, (float *)neg, (float *)pos,
                                workspace, workspace_bytes, st, t_lo, t_hi);
    }
    if (p->dtype == TNMF_F32)
        return generic_gradient_w<float>(g, (const float *)V, (const float *)R, (const float *)H, (float *)neg,
                                         (float *)pos, st, t_lo, t_hi);
    return generic_gradient_w<double>(g, (const double *)V, (const double *)R, (const double *)H, (double *)neg,
                                      (double *)pos, st, t_lo, t_hi);
}

int tnmf_update_w(const tnmf_problem *p, void *W, const void *neg, const void *pos, double eps, void *stream) {
    Geo g;
    int s = make_geo(p, g);
    if (s) return s;
    if (!W || !neg || !pos) return TNMF_EINVAL;
    cudaStream_t st = (cudaStream_t)stream;
    if (p->dtype == TNMF_F32) return update_w<float>(g, (float *)W, (const float *)neg, (const float *)pos, eps, st);
    return update_w<double>(g, (double *)W, (const double *)neg, (const double *)pos, eps, st);
}

size_t tnmf_peer_buffer_bytes(const tnmf_problem *p, int32_t world) {
    Geo g;
    if (make_geo(p, g, false) || world < 1 || world > TNMF_MAX_PEERS) return 0;
    return peer_buffer_bytes(g, p->dtype, world);
}

int tnmf_allreduce_update_w(const tnmf_problem *p, void *W, const void *grad, const tnmf_peer_world *peers, void *state,
                            double eps, void *stream) {
    Geo g;
    int s = make_geo(p, g, false);
    if (s) return s;
    if (!W || !grad || !peers || !state) return TNMF_EINVAL;
    if (peers->world < 1 || peers->world > TNMF_MAX_PEERS || peers->rank < 0 || peers->rank >= peers->world) return TNMF_EINVAL;
    for (int r = 0; r < peers->world; ++r)
        if (!peers->buffers[r]) return TNMF_EINVAL;
    cudaStream_t st = (cudaStream_t)stream;
    if (p->dtype == TNMF_F32)
        return allreduce_update_w<float>(g, p->dtype, (float *)W, (const float *)grad, peers, (unsigned *)state, eps, st);
    return allreduce_update_w<double>(g, p->dtype, (double *)W, (const double *)grad, peers, (unsigned *)state, eps, st);
}

int tnmf_normalize(int32_t dtype, void *arr, int64_t outer, int64_t len, int64_t inner, void *stream) {
    if (!arr || outer < 1 || len < 1 || inner < 1) return TNMF_EINVAL;
    cudaStream_t st = (cudaStream_t)stream;
    if (dtype == TNMF_F32) return normalize_axis<float>((float *)arr, outer, len, inner, st);
    if (dtype == TNMF_F64) return normalize_axis<double>((double *)arr, outer, len, inner, st);
    return TNMF_EUNSUPPORTED;
}

int tnmf_convolve_1d(int32_t dtype, const void *in, void *out, int64_t outer, int64_t len, int64_t inner,
                     const double *taps, int32_t n_taps, void *stream) {
    if (!in || !out || in == out || !taps || outer < 0 || len < 1 || inner < 1) return TNMF_EINVAL;
    if (outer == 0) return TNMF_OK;
    cudaStream_t st = (cudaStream_t)stream;
    if (dtype == TNMF_F32)
        return convolve_axis<float>((const float *)in, (float *)out, outer, len, inner, taps, n_taps, st);
    if (dtype == TNMF_F64)
        return convolve_axis<double>((const double *)in, (double *)out, outer, len, inner, taps, n_taps, st);
    return TNMF_EUNSUPPORTED;
}

int tnmf_sum_atoms(int32_t dtype, const void *G, void *Gsum, int64_t n_samples, int64_t n_atoms, int64_t inner,
                   void *stream) {
    if (!G || !Gsum || n_samples < 0 || n_atoms < 1 || inner < 1) return TNMF_EINVAL;
    if (n_samples == 0) return TNMF_OK;
    cudaStream_t st = (cudaStream_t)stream;
    if (dtype == TNMF_F32) return sum_atoms<float>((const float *)G, (float *)Gsum, n_samples, n_atoms, inner, st);
    if (dtype == TNMF_F64) return sum_atoms<double>((const double *)G, (double *)Gsum, n_samples, n_atoms, inner, st);
    return TNMF_EUNSUPPORTED;
}

int tnmf_fp32_peak_probe(void *sink, int32_t iterations, double *flops_out, void *stream) {
    if (!sink || iterations < 1) return TNMF_EINVAL;
    return fp32_peak_probe(sink, iterations, flops_out, (cudaStream_t)stream);
}

}  // extern "C"
