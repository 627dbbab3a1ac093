// Tensor-core (tcgen05, 3xTF32) reconstruction with the ACTIVATIONS AS A ROW RING IN TENSOR MEMORY
//   R[n,c,y,x] = sum_m sum_{ay,ax} W[m,c,ay,ax] * Hext[n,m,y+offy-ay,x+offx-ax]      (tnmf/backends/_Backend.py:120-122,
// NumPy.py:122-132), optionally fused with the energy 0.5*sum (V-R)^2 (tnmf/backends/_Backend.py:127-130).
//
// tc_recon.cu contracts over (atom, a_x) per SOURCE row and pays for it with 66 small MMAs whose 4 KB activation operand
// comes out of shared memory every time (44 clk each whatever their arithmetic).  Here the contraction runs over
// (atom row, atom) per OUTPUT row:
//   * a CTA owns 128 consecutive columns of the flattened [N x VW] space of virtual source columns, VW = DX + AX - 1 (virtual
//     column vv of a sample is the source column vv + offx - (AX-1); columns outside [0, TX) are the zero padding of 'full');
//   * the A operand is a RING of activation rows in TENSOR MEMORY: lane = column, 32-bit TMEM column = (ring slot, atom), hi
//     and lo halves.  An output row y needs the AY source rows y+offy-ay; when y advances ONE new row is written (each thread
//     loads the M activations of its column straight from global memory, splits them and issues two tcgen05.st) - no
//     shared-memory staging, no im2col, and the MMA's A operand costs no shared-memory bandwidth at all;
//   * B_ay[(c, ax), m] = W[m, c, ay, ax], resident in shared memory for every ay; the ring slot of source row ty pairs with
//     the matrix of ay = y + offy - ty: only a descriptor address changes from row to row;
//   * P[vv, (c, ax)] = sum_ay sum_m A[vv, (slot(ay), m)] * B_ay[(c, ax), m]:  AY * ceil(M/8) * 3 MMAs of M=128, N = roundup(C*AX, 16),
//     K=8 into a fresh TMEM buffer - with A in tensor memory they run at N/2 clk each (24 clk at N = 48; tools/tc_probe2.cu);
//   * the epilogue folds the a_x axis (col2im along x): R[c, y, x] = sum_ax P[x + AX-1 - ax, (c, ax)].  The four epilogue
//     warps move P through a [(c, ax)][column] array in shared memory (conflict-free both ways) and every thread sums the
//     AX entries of its output column; 2 * C * AX shared-memory words per output against 2 * M * AY * AX * C flops.
// Neighbouring tiles overlap by AX - 1 columns (a tile produces the 128 - (AX-1) outputs whose windows it holds completely).
// 3xTF32: hi*hi + lo*hi + hi*lo, FP32 accumulation in TMEM, one accumulation chain per output row (no long chains).
//
// Roles (576 threads): warps 0-7 write the ring (warp w: lane quarter w % 4, atom half w / 4; next row prefetched into
// registers); warps 8 and 9 issue the MMAs of alternate output rows (converged warps, one election per row, operands in
// uniform registers) - the tensor pipe queues only two or three MMAs, so whatever one warp spends between two rows (barrier
// waits, commits, descriptor arithmetic: ~900 clk against 1584 clk of MMAs, measured) is only hidden while the other warp
// keeps issuing; every P buffer is written by one warp, so the order of accumulation stays fixed.  Both warps walk ALL rows
// and both commit on every ring-slot release (a_free counts two arrivals: a slot is rewritten only when the MMAs of both
// warps that read it are done).  Warps 10-17 are two epilogue groups (thread = column = TMEM lane) serving alternate rows.
// mbarriers: a_full/a_free per ring slot, p_full/p_free per P buffer.
#include "tc_common.cuh"

namespace tnmf {
namespace tc {
namespace rct {

using tiled::ceil_div;
using tiled::Geo2;
using tiled::round_up;

constexpr int kTile = 128;
constexpr int kIssuers = 2;             // MMA-issuing warps: output row g belongs to warp g % 2
constexpr int kEpiGroups = 2;           // epilogue groups of 4 warps: output row g belongs to group g % 2
constexpr int kThreads = 32 * (8 + kIssuers + 4 * kEpiGroups);
constexpr int kRingMax = 32;
constexpr int kBufMax = 4;
constexpr int kMaxSmem = 226 * 1024;
constexpr int kAtomsPerThread = 16;     // most ring columns one writing thread takes per row (half of the padded atoms)

struct Plan {
    int KM, ksteps;                 // atoms padded to a multiple of 8
    int NU, NP;                     // C * AX and its padding to a multiple of 16 (MMA N)
    int VW, S;                      // virtual columns per sample, new output columns per tile
    int RS, NBUF, p_col0;           // ring slots, P buffers, first TMEM column of the P buffers
    int b_floats;                   // floats of ONE of the hi / lo halves of the atom operand
    int tiles;
    long long total, quota, units;  // tile-rows of the problem, tile-rows per CTA, grid * (most segments of a CTA)
    int grid;
    size_t smem;
};

struct Args {
    const float *W, *H, *V;
    float *R;
    double *epart;                  // grid * 8 partial energies (or null)
};

bool make_plan(const Geo2 &g, Plan &p) {
    p = Plan();
    if (g.C < 1 || g.AY < 1 || g.AX < 1 || g.AX > 64) return false;
    p.KM = round_up(g.M, 8);
    if (p.KM > 2 * kAtomsPerThread || (long long)kAtomsPerThread * g.hsm >= (1ll << 31)) return false;
    p.ksteps = p.KM / 8;
    p.NU = g.C * g.AX;
    p.NP = round_up(p.NU, 16);
    if (p.NP > 256) return false;
    // TMEM: ring of RS >= AY + 2 slots (spares: the next row is written while the current one is multiplied) x KM columns
    // x {hi, lo}, then 2..4 P buffers
    p.RS = g.AY + 2;                                        // + 1: written ahead, + 1: the releases of an issuing warp lag a row
    if (2 * p.RS * p.KM + 2 * p.NP > 512) return false;
    p.NBUF = (512 - 2 * p.RS * p.KM) / p.NP;
    if (p.NBUF > kBufMax) p.NBUF = kBufMax;
    // even: a P buffer then always belongs to the same issuing warp and the same epilogue group.  A barrier watched by
    // alternating waiters would be watched every other phase only, and a parity wait cannot tell phase u from phase u - 2.
    p.NBUF &= ~1;
    while (p.RS < kRingMax && 2 * (p.RS + 1) * p.KM + p.NBUF * p.NP <= 512) ++p.RS;
    p.p_col0 = 2 * p.RS * p.KM;
    p.VW = g.DX + g.AX - 1;
    p.S = kTile - (g.AX - 1);
    p.b_floats = g.AY * p.NP * p.KM;
    p.smem = (size_t)2 * p.b_floats * 4 + (size_t)kEpiGroups * 2 * p.NP * kTile * 4 + 1024;
    if (p.smem > (size_t)kMaxSmem) return false;
    const long long cols = (long long)g.N * p.VW;
    if (cols <= 0 || cols >= (1ll << 31) - kTile) return false;
    p.tiles = (int)((cols + p.S - 1) / p.S);
    // Work split: the (tile, row) space is cut into `grid` equal LINEAR ranges, one per CTA (a range is a few row segments
    // of consecutive tiles) - every SM gets the same number of rows whatever the number of tiles (cfg2: 138 / 145 / 276
    // tiles on 148 SMs left 7 - 10 % of the SMs idle with whole-tile units).  A segment boundary costs AY - 1 extra source
    // rows, and there are at most two per CTA.
    const int sms = tma::sm_count();
    p.total = (long long)p.tiles * g.DY;
    p.quota = (p.total + sms - 1) / sms;
    const long long min_quota = g.DY < 8 ? g.DY : 8;
    if (p.quota < min_quota) p.quota = min_quota;
    p.grid = (int)((p.total + p.quota - 1) / p.quota);
    p.units = (long long)p.grid * ((p.quota + g.DY - 2) / g.DY + 1);
    return true;
}

struct Unit {
    int tile, y0, y1, ta, tb;       // output rows [y0, y1), real source rows [ta, tb] (rows outside [0, TY) are zero: skipped)
};
__device__ __forceinline__ Unit make_unit(long long u, const Geo2 &g, const Plan &p) {
    // unit u = segment u / grid of CTA u % grid (gridDim.x == p.grid); empty (y0 == y1) past the CTA's last segment
    Unit w;
    const long long b = u % p.grid, k = u / p.grid;
    const long long lo = b * p.quota, hi = min(lo + p.quota, p.total);
    w.tile = (int)(lo / g.DY + k);
    const long long t0 = (long long)w.tile * g.DY;
    const long long s0 = max(lo, t0), s1 = min(hi, t0 + g.DY);
    w.y0 = s1 > s0 ? (int)(s0 - t0) : 0;
    w.y1 = s1 > s0 ? (int)(s1 - t0) : 0;
    w.ta = max(w.y0 + g.offy - (g.AY - 1), 0);
    w.tb = min(w.y1 - 1 + g.offy, g.TY - 1);
    return w;
}

__device__ __forceinline__ void tmem_st4(unsigned addr, float a, float b, float c, float d) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {%1, %2, %3, %4};\n" ::"r"(addr), "r"(__float_as_uint(a)),
                 "r"(__float_as_uint(b)), "r"(__float_as_uint(c)), "r"(__float_as_uint(d))
                 : "memory");
}

// C: channels (compile time: the epilogue's sums live in registers); APT: atoms per ring-writing thread = KM / 2
template <int C, int APT>
__global__ void __launch_bounds__(kThreads, 1) recon_ts_kernel(const Geo2 g, const Plan p, const Args a) {
    extern __shared__ __align__(128) float smem[];
    __shared__ __align__(8) unsigned long long a_full[kRingMax], a_free[kRingMax], p_full[kBufMax], p_free[kBufMax], turn[kIssuers];
    __shared__ unsigned tmem_base_s;
    const int tid = threadIdx.x, warp = __shfl_sync(0xffffffffu, tid >> 5, 0), lane = tid & 31;
    const int KM = p.KM, AY = g.AY, AX = g.AX, RS = p.RS, NP = p.NP, NU = p.NU;
    float *b_hi = smem, *b_lo = smem + p.b_floats;
    float *psm = b_lo + p.b_floats;                             // [group][2][NP][128]: P of one output row, (c, ax)-major

    if (tid == 0) {
        for (int s = 0; s < kRingMax; ++s) { mbar_init(&a_full[s], 8); mbar_init(&a_free[s], kIssuers); }
        for (int s = 0; s < kBufMax; ++s) { mbar_init(&p_full[s], 1); mbar_init(&p_free[s], 4); }
        for (int s = 0; s < kIssuers; ++s) mbar_init(&turn[s], 1);
        mbar_fence_init();
    }
    if (warp == 8) tmem_alloc(&tmem_base_s, 512);
    // atom operand: B[ay][n = c*AX + ax][k = m] = W[m, c, ay, ax]   (zero rows / atoms beyond)
    for (int idx = tid; idx < AY * NP * KM; idx += kThreads) {
        const int ay = idx / (NP * KM), r = idx - ay * (NP * KM);
        const int n = r / KM, m = r - n * KM;
        float v = 0.f;
        if (n < NU && m < g.M) {
            const int c = n / AX, ax = n - c * AX;
            v = a.W[(((long long)m * C + c) * AY + ay) * AX + ax];
        }
        float hi, lo;
        split_tf32(v, hi, lo);
        const size_t o = (size_t)ay * (NP * KM) + canon_offset_floats(n, m, NP);
        b_hi[o] = hi;
        b_lo[o] = lo;
    }
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const unsigned tmem_base = tmem_base_s;

    if (warp < 8) {
        // ------------------------------------ ring writers ------------------------------------
        const int quarter = warp & 3, half = warp >> 2;
        const int i = quarter * 32 + lane;                      // column of the tile = TMEM lane
        const int m_lo = half * APT;                            // this thread's atoms: [m_lo, m_lo + APT) of the KM padded ones
        const int m_valid = max(0, min(APT, g.M - m_lo));
        const unsigned t_lane = tmem_base + ((unsigned)(quarter * 32) << 16) + (unsigned)m_lo;
        int slot = 0;
        unsigned wraps = 0;
        TC_PROF_DECL(afree); TC_PROF_DECL(total);
#ifdef TNMF_TC_PROFILE
        prof_total = -clock64();
#endif
        for (long long u = blockIdx.x; u < p.units; u += gridDim.x) {
            const Unit w = make_unit(u, g, p);
            if (w.y0 >= w.y1) break;                            // past this CTA's last segment
            const long long F = (long long)w.tile * p.S + i;
            const int n = (int)(F / p.VW);
            const int v = (int)(F - (long long)n * p.VW) + g.offx - (AX - 1);
            const bool real = n < g.N && (unsigned)v < (unsigned)g.TX;
            // two rows are always in flight (the activations come from DRAM: ~1000 clk against ~1600 clk per row)
            const float *hnext = a.H + (real ? (long long)n * g.hsn + (long long)m_lo * g.hsm + v + (long long)w.ta * g.hsy : 0);
            const int mv = real ? m_valid : 0;
            float hva[APT], hvb[APT];
            auto load_row = [&](float (&hv)[APT]) {
#pragma unroll
                for (int e = 0; e < APT; ++e) hv[e] = e < mv ? __ldg(hnext + (unsigned)e * (unsigned)g.hsm) : 0.f;
                hnext += g.hsy;
            };
            auto write_row = [&](const float (&hv)[APT]) {
                if (wraps) TC_PROF_WAIT(afree, mbar_wait_backoff(&a_free[slot], (wraps - 1u) & 1u, 20));
                tc_fence_after();
                const unsigned t_hi = t_lane + (unsigned)(slot * KM), t_lo = t_hi + (unsigned)(RS * KM);
#pragma unroll
                for (int e = 0; e < APT; e += 4) {
                    float h0, h1, h2, h3, l0, l1, l2, l3;
                    split_tf32(hv[e], h0, l0); split_tf32(hv[e + 1], h1, l1);
                    split_tf32(hv[e + 2], h2, l2); split_tf32(hv[e + 3], h3, l3);
                    tmem_st4(t_hi + e, h0, h1, h2, h3);
                    tmem_st4(t_lo + e, l0, l1, l2, l3);
                }
                tmem_st_wait();
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(&a_full[slot]);
                if (++slot == RS) { slot = 0; ++wraps; }
            };
            if (w.ta <= w.tb) load_row(hva);
            if (w.ta + 1 <= w.tb) load_row(hvb);
            for (int ty = w.ta; ty <= w.tb; ty += 2) {
                write_row(hva);
                if (ty + 2 <= w.tb) load_row(hva);
                if (ty + 1 <= w.tb) {
                    write_row(hvb);
                    if (ty + 3 <= w.tb) load_row(hvb);
                }
            }
        }
#ifdef TNMF_TC_PROFILE
        prof_total += clock64();
        if (blockIdx.x == 0 && tid == 0) printf("recon_ts writers: total %lld  wait a_free %lld\n", prof_total, prof_afree);
#endif
    } else if (warp >= 8 + kIssuers) {
        // ------------------------------------ epilogue: fold the a_x axis ------------------------------------
        const int q = warp & 3, grp = (warp - (8 + kIssuers)) >> 2;
        const int i = q * 32 + lane;                            // TMEM lane = column of the tile
        const unsigned lane_base = tmem_base + ((unsigned)(q * 32) << 16) + (unsigned)p.p_col0;
        const long long plane = (long long)g.DY * g.DX;
        float *psm_g = psm + (size_t)grp * 2 * NP * kTile;
        double e_local = 0.0;
        int buf = 0;
        unsigned buf_wraps = 0, prow = 0, row = 0;              // row: output rows of this CTA so far (all groups)
        TC_PROF_DECL(pfull); TC_PROF_DECL(total); TC_PROF_DECL(bar); TC_PROF_DECL(ld); TC_PROF_DECL(fold);
#ifdef TNMF_TC_PROFILE
        prof_total = -clock64();
#endif
        for (long long u = blockIdx.x; u < p.units; u += gridDim.x) {
            const Unit w = make_unit(u, g, p);
            if (w.y0 >= w.y1) break;                            // past this CTA's last segment
            const long long F0 = (long long)w.tile * p.S + i;
            const int n = (int)(F0 / p.VW);
            const int xo = (int)(F0 - (long long)n * p.VW);
            const bool active = i < p.S && n < g.N && xo < g.DX;
            const long long obase = (long long)n * C * plane + xo;
            for (int y = w.y0; y < w.y1; ++y, ++row) {
                const int my_buf = buf;
                const unsigned my_par = buf_wraps & 1u;
                if (++buf == p.NBUF) { buf = 0; ++buf_wraps; }
                if ((int)(row % kEpiGroups) != grp) continue;
                float *ps = psm_g + (size_t)(prow & 1u) * NP * kTile;
                ++prow;
                TC_PROF_WAIT(pfull, mbar_wait_backoff(&p_full[my_buf], my_par, 20));
                tc_fence_after();
#ifdef TNMF_TC_PROFILE
                const long long t_l = clock64();
#endif
                if (NP <= 48) {
                    // all columns of the row in registers first: the P buffer goes back to its issuer after one TMEM round trip
                    float v[3][16];
#pragma unroll
                    for (int h = 0; h < 3; ++h)
                        if (16 * h < NP) tmem_ld16(lane_base + (unsigned)(my_buf * NP + 16 * h), v[h]);
                    tmem_ld_wait();
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(&p_free[my_buf]);
#pragma unroll
                    for (int h = 0; h < 3; ++h) {
                        const int cc = 16 * h;
                        float *pd = ps + cc * kTile + i;
                        if (cc + 16 <= NU) {
#pragma unroll
                            for (int k = 0; k < 16; ++k) pd[k * kTile] = v[h][k];
                        } else if (cc < NU) {
#pragma unroll
                            for (int k = 0; k < 16; ++k)
                                if (cc + k < NU) pd[k * kTile] = v[h][k];
                        }
                    }
                } else {
                    for (int c0 = 0; c0 < NP; c0 += 32) {             // two chunks of 16 columns in flight
                        float v[2][16];
                        tmem_ld16(lane_base + (unsigned)(my_buf * NP + c0), v[0]);
                        if (c0 + 16 < NP) tmem_ld16(lane_base + (unsigned)(my_buf * NP + c0 + 16), v[1]);
                        tmem_ld_wait();
#pragma unroll
                        for (int h = 0; h < 2; ++h) {
                            const int cc = c0 + 16 * h;
                            float *pd = ps + cc * kTile + i;
                            if (cc + 16 <= NU) {
#pragma unroll
                                for (int k = 0; k < 16; ++k) pd[k * kTile] = v[h][k];
                            } else if (cc < NU) {
#pragma unroll
                                for (int k = 0; k < 16; ++k)
                                    if (cc + k < NU) pd[k * kTile] = v[h][k];
                            }
                        }
                    }
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(&p_free[my_buf]);
                }
#ifdef TNMF_TC_PROFILE
                prof_ld += clock64() - t_l;
#endif
                TC_PROF_WAIT(bar, asm volatile("bar.sync %0, 128;\n" ::"r"(2 + grp) : "memory"));
#ifdef TNMF_TC_PROFILE
                const long long t_b = clock64();
                if (__float_as_uint(*(volatile float *)(ps + i)) == 0x7fc12345u) prof_fold += 1;     // first touch behind the barrier
                const long long t_f = clock64();
                prof_bar += t_f - t_b;
#endif
                if (active) {
                    // R[c, y, x] = sum_ax P[(c, ax)][i + AX-1 - ax].  All loads of a batch are issued before the first add: under
                    // the tensor core's operand traffic (it has priority on the shared-memory port) a dependent LDS round
                    // trip costs ~150 clk, and a loop of 4-wide chains made 15 of them per row (measured: 2300 clk per row).
                    float r[C];
#pragma unroll
                    for (int c = 0; c < C; ++c) r[c] = 0.f;
                    for (int ax0 = 0; ax0 < AX; ax0 += 16) {
                        float t[C][16];
#pragma unroll
                        for (int c = 0; c < C; ++c) {
                            const float *pc = ps + (size_t)(c * AX + ax0) * kTile + i + (AX - 1) - ax0;
#pragma unroll
                            for (int k = 0; k < 16; ++k) t[c][k] = (ax0 + k < AX) ? pc[k * (kTile - 1)] : 0.f;
                        }
#pragma unroll
                        for (int c = 0; c < C; ++c) {
#pragma unroll
                            for (int k = 0; k < 8; ++k) t[c][k] += t[c][k + 8];
#pragma unroll
                            for (int k = 0; k < 4; ++k) t[c][k] += t[c][k + 4];
                            r[c] += (t[c][0] + t[c][2]) + (t[c][1] + t[c][3]);
                        }
                    }
#pragma unroll
                    for (int c = 0; c < C; ++c) {
                        const long long o = obase + (long long)c * plane + (long long)y * g.DX;
                        if (a.R) a.R[o] = r[c];
                        if (a.V) {
                            const double d = (double)a.V[o] - (double)r[c];
                            e_local += d * d;
                        }
                    }
                }
#ifdef TNMF_TC_PROFILE
                prof_fold += clock64() - t_f;
#endif
            }
        }
#ifdef TNMF_TC_PROFILE
        prof_total += clock64();
        if (blockIdx.x == 0 && tid == (8 + kIssuers) * 32) printf("recon_ts epilogue: total %lld  wait p_full %lld  barrier %lld  tmem->smem %lld  fold %lld\n", prof_total, prof_pfull, prof_bar, prof_ld, prof_fold);
#endif
        if (a.epart) {                                          // one partial per epilogue warp
            for (int o = 16; o > 0; o >>= 1) e_local += __shfl_xor_sync(0xffffffffu, e_local, o);
            if (lane == 0) a.epart[(long long)blockIdx.x * (4 * kEpiGroups) + grp * 4 + q] = e_local;
        }
    } else {
        // ------------------------------------ MMA issuers: output row g -> warp 8 + g % 2 ------------------------------------
        const int x = warp - 8;
        const unsigned tmem_u = __shfl_sync(0xffffffffu, tmem_base, 0);
        const unsigned lbo_b = (unsigned)NP * 16;
        const unsigned desc_hi = (128u >> 4) | (1u << 14);      // SBO = 128, descriptor version 1
        // low descriptor words: start address (>> 4) + LBO field; the sums below never carry out of the 14 address bits
        const unsigned w_hi = __shfl_sync(0xffffffffu, (smem_u32(b_hi) >> 4) + ((lbo_b >> 4) << 16), 0);
        const unsigned w_lo = __shfl_sync(0xffffffffu, (smem_u32(b_lo) >> 4) + ((lbo_b >> 4) << 16), 0);
        const unsigned b_ay16 = ((unsigned)(NP * KM) * 4u) >> 4, b_step16 = (2 * lbo_b) >> 4;
        const unsigned idesc = idesc_tf32(kTile, NP);
        const unsigned lo_off = (unsigned)(RS * KM);
        const int ksteps = p.ksteps;
        int slot_new = 0, slot_first = 0, slot_rel = 0;         // next slot to be filled / first slot of the window / next to free
        unsigned par_new = 0;
        int buf = 0;
        unsigned buf_wraps = 0, row = 0;
        TC_PROF_DECL(afull); TC_PROF_DECL(pfree); TC_PROF_DECL(total); TC_PROF_DECL(issue); TC_PROF_DECL(turnw); TC_PROF_DECL(commit); TC_PROF_DECL(elect);
#ifdef TNMF_TC_PROFILE
        prof_total = -clock64();
#endif
        for (long long u = blockIdx.x; u < p.units; u += gridDim.x) {
            const Unit w = make_unit(u, g, p);
            if (w.y0 >= w.y1) break;                            // past this CTA's last segment
            int next_new = w.ta, first = w.ta, next_rel = w.ta;
            slot_first = slot_new;
            slot_rel = slot_new;
            for (int y = w.y0; y < w.y1; ++y, ++row) {
                const int my_buf = buf;
                const unsigned my_wraps = buf_wraps;
                if (++buf == p.NBUF) { buf = 0; ++buf_wraps; }
                const bool last_row = y + 1 == w.y1;
                // A warp touches the barriers only on its own rows (and on the last row of a unit, where the ring is handed
                // over): it catches up on the source rows that arrived meanwhile, and its slot releases lag one row behind
                // (the ring has the spare slot for it).  Rows of the other warp cost a few integer operations.
                if ((int)(row % kIssuers) != x && !last_row) continue;
                // (every output row meets at least one real source row in both modes: t_first <= t_last)
                const int t_last = min(w.tb, y + g.offy), t_first = max(w.ta, y + g.offy - (AY - 1));
                for (; next_new <= t_last; ++next_new) {
                    TC_PROF_WAIT(afull, mbar_wait(&a_full[slot_new], par_new));
                    if (++slot_new == RS) { slot_new = 0; par_new ^= 1u; }
                }
                for (; first < t_first; ++first)
                    if (++slot_first == RS) slot_first = 0;
                if ((int)(row % kIssuers) == x) {
                    if (my_wraps) TC_PROF_WAIT(pfree, mbar_wait(&p_free[my_buf], (my_wraps - 1u) & 1u));
                    // Take turns: this warp starts once the other one is half way through the previous row.  Left alone,
                    // the two warps fall into lockstep - they share the pipe evenly, finish together and then both do their
                    // bookkeeping while the pipe idles (measured: pipe busy 57 % of the time).
                    if (row > 0) TC_PROF_WAIT(turnw, mbar_wait(&turn[x], ((row - 1u) >> 1) & 1u));
                    tc_fence_after();
#ifdef TNMF_TC_PROFILE
                    const long long t_i = clock64();
#endif
                    const unsigned tp = tmem_u + (unsigned)(p.p_col0 + my_buf * NP);
                    if (elect_one()) {
                        // The issuing lane must hand the pipe an MMA every N/2 = 24 clk: nothing but uniform adds may stand
                        // between two of them.  The K steps are a compile-time count (KM = 2 * APT), the one non-accumulating
                        // MMA of the row is peeled off (a `fresh` flag inside the loop cost a vote and six moves per K step -
                        // ncu: tensor pipe 62 % active with the issuing warps never waiting), and the row is cut at its
                        // middle for the hand-over to the other warp instead of testing for it in every iteration.
                        constexpr int kSteps = APT / 4;
                        int s = slot_first;
                        unsigned bo = (unsigned)(y + g.offy - t_first) * b_ay16;    // matrix of ay = y + offy - ty
                        {
                            const unsigned ta_hi = tmem_u + (unsigned)(s * KM), ta_lo = ta_hi + lo_off;
                            mma_tf32_ts2<false>(tp, ta_hi, w_hi + bo, desc_hi, idesc);
                            mma_tf32_ts2<true>(tp, ta_lo, w_hi + bo, desc_hi, idesc);
                            mma_tf32_ts2<true>(tp, ta_hi, w_lo + bo, desc_hi, idesc);
#pragma unroll
                            for (int ks = 1; ks < kSteps; ++ks) {
                                const unsigned kb = bo + (unsigned)ks * b_step16;
                                mma_tf32_ts2<true>(tp, ta_hi + 8u * ks, w_hi + kb, desc_hi, idesc);
                                mma_tf32_ts2<true>(tp, ta_lo + 8u * ks, w_hi + kb, desc_hi, idesc);
                                mma_tf32_ts2<true>(tp, ta_hi + 8u * ks, w_lo + kb, desc_hi, idesc);
                            }
                            if (++s == RS) s = 0;
                            bo -= b_ay16;
                        }
#ifndef TNMF_RCT_TURN_DIV
#define TNMF_RCT_TURN_DIV 2
#endif
                        const int t_mid = max(t_first + (t_last - t_first + 1) / TNMF_RCT_TURN_DIV, t_first + 1);
                        auto rows = [&](int ty_a, int ty_b) {
                            for (int ty = ty_a; ty < ty_b; ++ty) {
                                const unsigned ta_hi = tmem_u + (unsigned)(s * KM), ta_lo = ta_hi + lo_off;
#pragma unroll
                                for (int ks = 0; ks < kSteps; ++ks) {
                                    const unsigned kb = bo + (unsigned)ks * b_step16;
                                    mma_tf32_ts2<true>(tp, ta_hi + 8u * ks, w_hi + kb, desc_hi, idesc);
                                    mma_tf32_ts2<true>(tp, ta_lo + 8u * ks, w_hi + kb, desc_hi, idesc);
                                    mma_tf32_ts2<true>(tp, ta_hi + 8u * ks, w_lo + kb, desc_hi, idesc);
                                }
                                if (++s == RS) s = 0;
                                bo -= b_ay16;
                            }
                        };
                        rows(t_first + 1, min(t_mid, t_last + 1));
                        mbar_arrive(&turn[x ^ 1]);                                  // the other warp may start on the next row
                        rows(t_mid, t_last + 1);
                    }
                    __syncwarp();
#ifdef TNMF_TC_PROFILE
                    const long long t_c = clock64();
                    prof_issue += t_c - t_i;
#endif
                    mma_commit_elect(&p_full[my_buf]);
#ifdef TNMF_TC_PROFILE
                    prof_commit += clock64() - t_c;
#endif
                }
#ifdef TNMF_TC_PROFILE
                const long long t_r = clock64();
#endif
                // Source rows no later output row of this unit reads: their slots may be rewritten once the MMAs that read
                // them are done.  BOTH warps commit (a_free counts two arrivals): each commit covers the committing warp's
                // own MMAs.
                const int rel_to = last_row ? w.tb + 1 : min(w.tb + 1, y + 1 + g.offy - (AY - 1));
                for (; next_rel < rel_to; ++next_rel) {
                    mma_commit_elect(&a_free[slot_rel]);
                    if (++slot_rel == RS) slot_rel = 0;
                }
#ifdef TNMF_TC_PROFILE
                prof_elect += clock64() - t_r;
#endif
            }
        }
#ifdef TNMF_TC_PROFILE
        prof_total += clock64();
        if (blockIdx.x == 0 && lane == 0 && x == 0)
            printf("recon_ts mma: total %lld  wait a_full %lld  wait p_free %lld  wait turn %lld  issuing %lld  commit p_full %lld  release commits %lld\n", prof_total, prof_afull, prof_pfree, prof_turnw, prof_issue, prof_commit, prof_elect);
#endif
        __syncwarp();
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 8) tmem_dealloc(tmem_base, 512);
}

template <int C, int APT>
static int launch2(const Geo2 &g, const Plan &p, const Args &a, cudaStream_t st) {
    auto kern = recon_ts_kernel<C, APT>;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, kMaxSmem);
    if (e != cudaSuccess) return status_from_cuda(e);
    kern<<<(unsigned)p.grid, kThreads, p.smem, st>>>(g, p, a);
    TNMF_CHECK_LAUNCH();
    return TNMF_OK;
}

template <int C>
static int launch(const Geo2 &g, const Plan &p, const Args &a, cudaStream_t st) {
    switch (p.KM / 2) {
        case 4: return launch2<C, 4>(g, p, a, st);
        case 8: return launch2<C, 8>(g, p, a, st);
        case 12: return launch2<C, 12>(g, p, a, st);
        case 16: return launch2<C, 16>(g, p, a, st);
        default: return TNMF_EUNSUPPORTED;
    }
}

}  // namespace rct
}  // namespace tc

// ---- dispatch ----------------------------------------------------------------------------------------------------------
bool tc_recon_ts_supported(const Geo &g, int dtype) {
    if (!tc::rank2_ok(g, dtype) || g.C > 4) return false;
    tc::rct::Plan p;
    return tc::rct::make_plan(tiled::make_geo2(g), p);
}

int tc_recon_ts_partials(const Geo &g) {
    tc::rct::Plan p;
    return tc::rct::make_plan(tiled::make_geo2(g), p) ? p.grid * 4 * tc::rct::kEpiGroups : 0;
}

int tc_reconstruct_ts(const Geo &g, const float *W, const float *H, float *R, const float *V, double *energy_partials,
                      int *n_partials, cudaStream_t st) {
    const tiled::Geo2 q = tiled::make_geo2(g);
    tc::rct::Plan p;
    if (!tc::rct::make_plan(q, p)) return TNMF_EUNSUPPORTED;
    tc::rct::Args a;
    a.W = W; a.H = H; a.V = V; a.R = R; a.epart = energy_partials;
    if (n_partials) *n_partials = p.grid * 4 * tc::rct::kEpiGroups;
    switch (g.C) {
        case 1: return tc::rct::launch<1>(q, p, a, st);
        case 2: return tc::rct::launch<2>(q, p, a, st);
        case 3: return tc::rct::launch<3>(q, p, a, st);
        case 4: return tc::rct::launch<4>(q, p, a, st);
        default: return TNMF_EUNSUPPORTED;
    }
}

}  // namespace tnmf
