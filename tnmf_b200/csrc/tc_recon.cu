// Tensor-core (tcgen05, 3xTF32) reconstruction  R[n,c,y,x] = sum_m sum_{ay,ax} W[m,c,ay,ax] * Hext[n,m,y+offy-ay,x+offx-ax]
// (tnmf/backends/_Backend.py:120-122, NumPy.py:122-132), optionally fused with the energy 0.5*sum (V-R)^2
// (tnmf/backends/_Backend.py:127-130).
//
// The only free index on the W side of this contraction is the channel, so an output-stationary GEMM has N = C.  The
// formulation here is INPUT-stationary and needs no im2col at all:
//   * a CTA owns 128 output columns (column J = n * DXP + x of the flattened [N x DXP] space, DXP = DX + AX - 1, so the
//     activation windows of different samples never meet) and walks down the SOURCE rows ty of H;
//   * the activation row tile is staged once as A[rho, m] (row = virtual position, K = atom, canonical K-major layout
//     whose rows sit 16 bytes apart): the operand of atom column ax is the SAME tile read from row AX-1-ax on - a shift
//     of the descriptor's start address, no copy;
//   * B_ax[(ay, c), m] = W[m, c, ay, ax] (N = roundup(AY*C, 16) rows, all AX of them resident in shared memory);
//   * per source row: Q[x, (ay, c)] = sum_ax sum_m A_ax[x, m] * B_ax[(ay, c), m]   - AX * ceil(M/8) * 3 MMAs of
//     M=128, N<=64, K=8 into one TMEM buffer (fresh per source row: no long truncating accumulation chains);
//   * the epilogue thread of a column keeps the AY output rows in flight in REGISTERS: it adds Q[.., (ay, c)] to the
//     partial sum of row y = ty - offy + ay, emits row ty - offy (complete) and shifts the ring by one row.
// 3xTF32: hi*hi + lo*hi + hi*lo, FP32 accumulation.  Bound: tcgen05 issue rate (N <= 64: every MMA sits on the
// per-instruction floor), which is why several warps issue alternate source rows into alternate TMEM buffers (each
// buffer is written by one warp only: the accumulation order is fixed).
//
// Roles (448 threads): warps 0-7 stage the activation rows (global -> hi/lo -> shared), warps 8-11 epilogue (thread =
// output column = TMEM lane), warps 12.. issue the MMAs (source row g belongs to issuing warp g % kIssuers).  mbarriers: a_full/a_empty per
// operand stage, d_full/d_free per TMEM buffer.
#include "tc_common.cuh"

namespace tnmf {
namespace tc {
namespace rc {

using tiled::ceil_div;
using tiled::Geo2;
using tiled::round_up;

constexpr int kTile = 128;
constexpr int kWorkers = 256;
#ifndef TNMF_RC_ISSUERS
#define TNMF_RC_ISSUERS 4
#endif
constexpr int kIssuers = TNMF_RC_ISSUERS;    // MMA-issuing warps: source row g belongs to warp g % kIssuers
constexpr int kThreads = 32 * (12 + kIssuers);
constexpr int kMaxStages = 6;
constexpr int kBufs = 8;            // TMEM buffers of 64 columns
constexpr int kMaxSmem = 226 * 1024;
constexpr int kChunkMax = 6;        // 16-byte chunks of an activation stage per worker

struct Plan {
    int KM, ksteps;                 // atoms padded to a multiple of 8
    int NP;                         // AY * C padded to a multiple of 16 (MMA N)
    int DXP, RWS, RWSp;             // padded columns per sample, staged rows, rounded to 8
    int nchunk;
    int tiles, rblocks, rows_per_block;
    long long units;
    int n_stages, stage_floats, b_floats;   // floats of ONE of the hi / lo halves
    int n_issuers;                  // issuing warps in use: at most n_stages (see the issuer loop)
    int grid;
    size_t smem;
};

struct Args {
    const float *W, *H, *V;
    float *R;
    double *epart;                  // grid * 4 partial energies (or null)
};

bool make_plan(const Geo2 &g, Plan &p) {
    p = Plan();
    if (g.C < 1 || g.C > 4 || g.AY < 1 || g.AY > 16) return false;     // register ring of AY*C <= 64 partial sums
    p.NP = round_up(g.AY * g.C, 16);
    if (p.NP > 64) return false;
    p.KM = round_up(g.M, 8);
    if (p.KM > 64) return false;
    p.ksteps = p.KM / 8;
    p.DXP = g.DX + g.AX - 1;
    p.RWS = kTile + g.AX - 1;
    p.RWSp = round_up(p.RWS, 8);
    p.stage_floats = p.RWSp * p.KM;
    p.b_floats = g.AX * p.NP * p.KM;
    p.nchunk = ceil_div(p.RWSp * (p.KM / 4), kWorkers);
    if (p.nchunk > kChunkMax) return false;
    const size_t fixed = (size_t)2 * p.b_floats * 4 + 1024;
    if (fixed + 2 * (size_t)2 * p.stage_floats * 4 > (size_t)kMaxSmem) return false;
    p.n_stages = (int)(((size_t)kMaxSmem - fixed) / ((size_t)2 * p.stage_floats * 4));
    if (p.n_stages > kMaxStages) p.n_stages = kMaxStages;
    p.smem = fixed + (size_t)p.n_stages * 2 * p.stage_floats * 4;
    p.n_issuers = p.n_stages < kIssuers ? p.n_stages : kIssuers;
    const long long cols = (long long)g.N * p.DXP;
    if (cols <= 0 || cols >= (1ll << 31) - kTile) return false;
    p.tiles = (int)((cols + kTile - 1) / kTile);
    const int sms = tma::sm_count();
    double best = -1;
    for (int rb = 1; rb <= g.DY && rb <= 64; ++rb) {
        const int rows = ceil_div(g.DY, rb);
        if (ceil_div(g.DY, rows) != rb) continue;
        const long long units = (long long)p.tiles * rb;
        const double waves = (double)((units + sms - 1) / sms);
        const double cost = waves * (rows + (g.AY - 1) + 1.0);     // a row block re-reads AY-1 source rows
        if (best < 0 || cost < best * 0.999) { best = cost; p.rblocks = rb; p.rows_per_block = rows; }
    }
    p.units = (long long)p.tiles * p.rblocks;
    p.grid = (int)(p.units < sms ? p.units : sms);
    return true;
}

struct Unit {
    int tile, y0, y1, t_lo, t_hi;   // output rows [y0, y1), source rows [t_lo, t_hi] (may leave [0, TY): those are zero)
};
__device__ __forceinline__ Unit make_unit(long long u, const Geo2 &g, const Plan &p) {
    Unit w;
    const int rb = (int)(u / p.tiles);
    w.tile = (int)(u - (long long)rb * p.tiles);
    w.y0 = rb * p.rows_per_block;
    w.y1 = min(g.DY, w.y0 + p.rows_per_block);
    w.t_lo = w.y0 + g.offy - (g.AY - 1);
    w.t_hi = w.y1 - 1 + g.offy;
    return w;
}

template <int C, int NP>
__global__ void __launch_bounds__(kThreads, 1) recon_tc_kernel(const Geo2 g, const Plan p, const Args a) {
    extern __shared__ __align__(128) float smem[];
    __shared__ __align__(8) unsigned long long a_full[kMaxStages], a_empty[kMaxStages], d_full[kBufs], d_free[kBufs];
    __shared__ unsigned tmem_base_s;
    // warp index out of a shuffle: warp-uniform role branches, MMA operands in uniform registers (see tc_gradw_ts.cu)
    const int tid = threadIdx.x, warp = __shfl_sync(0xffffffffu, tid >> 5, 0), lane = tid & 31;
    const int KM = p.KM, AY = g.AY, AX = g.AX;
    float *b_hi = smem, *b_lo = smem + p.b_floats;
    float *stages = b_lo + p.b_floats;                          // [stage][hi, lo][stage_floats]

    if (tid == 0) {
        for (int s = 0; s < p.n_stages; ++s) { mbar_init(&a_full[s], kWorkers); mbar_init(&a_empty[s], 1); }
        for (int s = 0; s < kBufs; ++s) { mbar_init(&d_full[s], 1); mbar_init(&d_free[s], kTile); }
        mbar_fence_init();
    }
    if (warp == 12) tmem_alloc(&tmem_base_s, 512);
    // atom operand of every atom column: B[ax][n = ay*C + c][k = m] = W[m, c, ay, ax]   (zero rows / atoms beyond)
    for (int idx = tid; idx < AX * NP * KM; idx += kThreads) {
        const int ax = idx / (NP * KM), r = idx - ax * (NP * KM);
        const int n = r / KM, m = r - n * KM;
        float v = 0.f;
        if (n < AY * C && m < g.M) {
            const int ay = n / C, c = n - ay * C;
            v = a.W[(((long long)m * C + c) * AY + ay) * AX + ax];
        }
        float hi, lo;
        split_tf32(v, hi, lo);
        const size_t o = (size_t)ax * (NP * KM) + canon_offset_floats(n, m, NP);
        b_hi[o] = hi;
        b_lo[o] = lo;
    }
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const unsigned tmem_base = tmem_base_s;

    if (warp < 8) {
        // ------------------------------------ workers: activation row tiles ------------------------------------
        // chunk q = tid + 256 e -> (atom group kc, staged row rho); fixed for the kernel
        const int n_rows = p.RWSp, n_chunks = n_rows * (KM / 4);
        long long g_row = 0;                                    // valid source rows staged so far
        for (long long u = blockIdx.x; u < p.units; u += gridDim.x) {
            const Unit w = make_unit(u, g, p);
            // element offset of (row rho, atom 4 kc) in source row 0, or -1: zero (gap / outside the sample)
            long long hoff[kChunkMax];
#pragma unroll
            for (int e = 0; e < kChunkMax; ++e) {
                hoff[e] = -1;
                const int q = tid + kWorkers * e;
                if (e < p.nchunk && q < n_chunks) {
                    const int kc = q / n_rows, rho = q - kc * n_rows;
                    const long long P = (long long)w.tile * kTile + rho;
                    const int n = (int)(P / p.DXP);
                    const int tx = (int)(P - (long long)n * p.DXP) + g.offx - (AX - 1);
                    if (rho < p.RWS && n < g.N && (unsigned)tx < (unsigned)g.TX && 4 * kc < g.M)
                        hoff[e] = (long long)n * g.hsn + (long long)(4 * kc) * g.hsm + tx;
                }
            }
            float4 hv[kChunkMax];
            auto load_row = [&](int ty) {
#pragma unroll
                for (int e = 0; e < kChunkMax; ++e) {
                    hv[e] = make_float4(0.f, 0.f, 0.f, 0.f);
                    if (hoff[e] >= 0) {
                        const int m0 = 4 * ((tid + kWorkers * e) / n_rows);
                        const float *src = a.H + hoff[e] + (long long)ty * g.hsy;
                        hv[e].x = src[0];
                        if (m0 + 1 < g.M) hv[e].y = src[g.hsm];
                        if (m0 + 2 < g.M) hv[e].z = src[2 * g.hsm];
                        if (m0 + 3 < g.M) hv[e].w = src[3 * g.hsm];
                    }
                }
            };
            const int ta = max(w.t_lo, 0), tb = min(w.t_hi, g.TY - 1);
            if (ta <= tb) load_row(ta);
            for (int ty = ta; ty <= tb; ++ty) {
                const int st = (int)(g_row % p.n_stages);
                if (g_row >= p.n_stages) mbar_wait_backoff(&a_empty[st], (unsigned)(((g_row / p.n_stages) - 1) & 1), 40);
                float *d_hi = stages + (size_t)st * 2 * p.stage_floats, *d_lo = d_hi + p.stage_floats;
#pragma unroll
                for (int e = 0; e < kChunkMax; ++e) {
                    const int q = tid + kWorkers * e;
                    if (e < p.nchunk && q < n_chunks) {
                        const int kc = q / n_rows, rho = q - kc * n_rows;
                        float4 hi, lo;
                        split_tf32(hv[e].x, hi.x, lo.x); split_tf32(hv[e].y, hi.y, lo.y);
                        split_tf32(hv[e].z, hi.z, lo.z); split_tf32(hv[e].w, hi.w, lo.w);
                        const size_t o = (size_t)(rho >> 3) * 32 + (size_t)kc * (n_rows * 4) + (size_t)(rho & 7) * 4;
                        *reinterpret_cast<float4 *>(d_hi + o) = hi;
                        *reinterpret_cast<float4 *>(d_lo + o) = lo;
                    }
                }
                if (ty < tb) load_row(ty + 1);                      // in flight while the MMAs of this row run
                fence_proxy_async();
                mbar_arrive(&a_full[st]);
                ++g_row;
            }
        }
    } else if (warp < 12) {
        // ------------------------------------ epilogue: register ring of AY output rows ------------------------------------
        const int i = tid - kWorkers;
        const unsigned lane_base = (unsigned)((warp & 3) * 32) << 16;
        const long long plane = (long long)g.DY * g.DX;
        double e_local = 0.0;
        long long g_row = 0;
        for (long long u = blockIdx.x; u < p.units; u += gridDim.x) {
            const Unit w = make_unit(u, g, p);
            const long long J = (long long)w.tile * kTile + i;
            const int n = (int)(J / p.DXP);
            const int xo = (int)(J - (long long)n * p.DXP);
            const bool active = n < g.N && xo < g.DX;
            const long long obase = (long long)n * C * plane + xo;
            float ring[NP];                                     // ring[ay*C + c]: partial sum of output row ty - offy + ay
#pragma unroll
            for (int k = 0; k < NP; ++k) ring[k] = 0.f;
            for (int ty = w.t_lo; ty <= w.t_hi; ++ty) {
                if (ty >= 0 && ty < g.TY) {
                    const int buf = (int)(g_row % kBufs);
                    mbar_wait_backoff(&d_full[buf], (unsigned)((g_row / kBufs) & 1), 40);
                    tc_fence_after();
#pragma unroll
                    for (int c0 = 0; c0 < NP; c0 += 16) {
                        float v[16];
                        tmem_ld16(tmem_base + lane_base + (unsigned)(buf * 64 + c0), v);
                        tmem_ld_wait();
#pragma unroll
                        for (int k = 0; k < 16; ++k) ring[c0 + k] += v[k];
                    }
                    tc_fence_before();
                    mbar_arrive(&d_free[buf]);
                    ++g_row;
                }
                // output row ty - offy has received its last contribution (ay = 0)
                const int y = ty - g.offy;
                if (active && y >= w.y0 && y < w.y1) {
#pragma unroll
                    for (int c = 0; c < C; ++c) {
                        const long long o = obase + (long long)c * plane + (long long)y * g.DX;
                        if (a.R) a.R[o] = ring[c];
                        if (a.V) {
                            const double d = (double)a.V[o] - (double)ring[c];
                            e_local += d * d;
                        }
                    }
                }
#pragma unroll
                for (int k = 0; k < NP - C; ++k) ring[k] = ring[k + C];
#pragma unroll
                for (int k = NP - C; k < NP; ++k) ring[k] = 0.f;
            }
        }
        if (a.epart) {                                          // one partial per epilogue warp
            for (int o = 16; o > 0; o >>= 1) e_local += __shfl_xor_sync(0xffffffffu, e_local, o);
            if (lane == 0) a.epart[(long long)blockIdx.x * 4 + (warp & 3)] = e_local;
        }
    } else {
        // ------------------------------------ MMA issuers: source row g -> warp 12 + g % kIssuers ------------------------------------
        const int x = warp - 12;
        const unsigned lbo_a = (unsigned)p.RWSp * 16, lbo_b = (unsigned)NP * 16;
        const unsigned desc_hi = (128u >> 4) | (1u << 14);                      // SBO, descriptor version 1
        const unsigned a_lo_word = ((lbo_a >> 4) << 16), b_lo_word = ((lbo_b >> 4) << 16);
        const unsigned b_hi16 = __shfl_sync(0xffffffffu, smem_u32(b_hi) >> 4, 0), b_lo16 = __shfl_sync(0xffffffffu, smem_u32(b_lo) >> 4, 0);
        const unsigned b16[3] = {b_hi16, b_hi16, b_lo16};
        const unsigned stage_addr0 = __shfl_sync(0xffffffffu, smem_u32(stages), 0);
        const unsigned tmem_u = __shfl_sync(0xffffffffu, tmem_base, 0);
        const unsigned a_step16 = (2 * lbo_a) >> 4, b_step16 = (2 * lbo_b) >> 4, b_ax16 = ((unsigned)(NP * KM) * 4u) >> 4;
        const unsigned idesc = idesc_tf32(kTile, NP);
        long long g_row = 0;
        for (long long u = blockIdx.x; u < p.units; u += gridDim.x) {
            const Unit w = make_unit(u, g, p);
            const int ta = max(w.t_lo, 0), tb = min(w.t_hi, g.TY - 1);
            for (int ty = ta; ty <= tb; ++ty, ++g_row) {
                // A warp that skips rows only ever tests the parity of a barrier; that is the right phase only while it is
                // at most one phase away, i.e. while the rows it skips fit into the stage ring: n_issuers <= n_stages.
                if ((int)(g_row % p.n_issuers) != x) continue;
                const int st = (int)(g_row % p.n_stages), buf = (int)(g_row % kBufs);
                if (g_row >= kBufs) mbar_wait(&d_free[buf], (unsigned)(((g_row / kBufs) - 1) & 1));
                mbar_wait(&a_full[st], (unsigned)((g_row / p.n_stages) & 1));
                tc_fence_after();
                const unsigned a_hi16 = (stage_addr0 + (unsigned)st * 2u * (unsigned)p.stage_floats * 4u) >> 4;
                const unsigned a_addr16[3] = {a_hi16, a_hi16 + (((unsigned)p.stage_floats * 4u) >> 4), a_hi16};
                const unsigned tbuf = tmem_u + (unsigned)(buf * 64);
                if (elect_one()) {                  // one election per source row: operands go to uniform registers once
                    unsigned acc = 0u;
                    for (int ax = 0; ax < AX; ++ax) {
                        const unsigned shift16 = (unsigned)(AX - 1 - ax);   // operand rows start AX-1-ax rows into the tile
                        for (int ks = 0; ks < p.ksteps; ++ks) {
#pragma unroll
                            for (int t = 0; t < 3; ++t) {
                                const unsigned long long da = ((unsigned long long)desc_hi << 32) |
                                                              (a_lo_word | (a_addr16[t] + shift16 + ks * a_step16));
                                const unsigned long long db = ((unsigned long long)desc_hi << 32) |
                                                              (b_lo_word | (b16[t] + ax * b_ax16 + ks * b_step16));
                                mma_tf32(tbuf, da, db, idesc, acc);
                                acc = 1u;
                            }
                        }
                    }
                }
                __syncwarp();
                mma_commit_elect(&a_empty[st]);
                mma_commit_elect(&d_full[buf]);
            }
        }
        __syncwarp();
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 12) tmem_dealloc(tmem_base, 512);
}

template <int C, int NP>
static int launch(const Geo2 &g, const Plan &p, const Args &a, cudaStream_t st) {
    auto kern = recon_tc_kernel<C, NP>;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, kMaxSmem);
    if (e != cudaSuccess) return status_from_cuda(e);
    kern<<<(unsigned)p.grid, kThreads, p.smem, st>>>(g, p, a);
    TNMF_CHECK_LAUNCH();
    return TNMF_OK;
}

}  // namespace rc
}  // namespace tc

// ---- dispatch ----------------------------------------------------------------------------------------------------------
bool tc_recon_supported(const Geo &g, int dtype) {
    if (!tc::rank2_ok(g, dtype)) return false;
    tc::rc::Plan p;
    return tc::rc::make_plan(tiled::make_geo2(g), p);
}

int tc_recon_partials(const Geo &g) {
    tc::rc::Plan p;
    return tc::rc::make_plan(tiled::make_geo2(g), p) ? p.grid * 4 : 0;
}

int tc_reconstruct(const Geo &g, const float *W, const float *H, float *R, const float *V, double *energy_partials,
                   int *n_partials, cudaStream_t st) {
    const tiled::Geo2 q = tiled::make_geo2(g);
    tc::rc::Plan p;
    if (!tc::rc::make_plan(q, p)) return TNMF_EUNSUPPORTED;
    tc::rc::Args a;
    a.W = W; a.H = H; a.V = V; a.R = R; a.epart = energy_partials;
    if (n_partials) *n_partials = p.grid * 4;
#define TNMF_RC_CASE(c, np) if (g.C == c && p.NP == np) return tc::rc::launch<c, np>(q, p, a, st);
    TNMF_RC_CASE(1, 16)
    TNMF_RC_CASE(2, 16) TNMF_RC_CASE(2, 32)
    TNMF_RC_CASE(3, 16) TNMF_RC_CASE(3, 32) TNMF_RC_CASE(3, 48)
    TNMF_RC_CASE(4, 16) TNMF_RC_CASE(4, 32) TNMF_RC_CASE(4, 48) TNMF_RC_CASE(4, 64)
#undef TNMF_RC_CASE
    return TNMF_EUNSUPPORTED;
}

}  // namespace tnmf
