// Tensor-core (tcgen05, 3xTF32) reconstruction for NARROW atoms: the OUTPUT ROWS ARE A RING OF ACCUMULATORS IN TENSOR MEMORY
//   R[n,c,y,x] = sum_m sum_{ay,ax} W[m,c,ay,ax] * Hext[n,m,y+offy-ay,x+offx-ax]      (tnmf/backends/_Backend.py:120-122,
// NumPy.py:122-132), optionally fused with the energy 0.5*sum (V-R)^2 (tnmf/backends/_Backend.py:127-130).
//
// tc_recon_ts.cu keeps a ring of A_y activation rows in tensor memory (2 * (A_y + 2) * atoms columns) and contracts over
// (atom row, atom) per OUTPUT row with MMAs of N = roundup(C * A_x, 16).  With one channel and many atoms (BASELINE config
// 3: C = 1, 32 atoms of 15 x 15) the ring does not fit the 512 columns and the MMAs would have N = 16.  Here the roles are
// swapped - the kernel is SOURCE-row stationary:
//   * a CTA owns 128 consecutive columns of the flattened [N x VW] space of virtual source columns (VW = DX + AX - 1, as in
//     tc_recon_ts.cu) and walks down the source rows ty of H;
//   * the A operand is ONE activation row in TENSOR MEMORY (lane = column, 32-bit TMEM column = atom; hi and lo halves),
//     written by the thread that owns the column straight from global memory, in a ring of 2..4 stages;
//   * B[(ay, c, ax), m] = W[m, c, ay, ax] for ALL atom rows is resident in shared memory (rows ordered by ay);
//   * source row ty contributes to the A_y output rows y = ty - offy + ay at once:
//         P_y[vv, (c, ax)] += sum_m A_ty[vv, m] * B[(ay = y + offy - ty, c, ax), m]
//     is ONE accumulating MMA of M = 128, N = (rows in the window) * NP <= 256, K = 8 per K step (two when the window wraps
//     around the ring), into a ring of RSD >= A_y + 1 output-row accumulators of NP = roundup(C * A_x, 16) TMEM columns;
//     consecutive output rows are consecutive ring slots AND consecutive row blocks of B, so only two addresses change;
//   * when its last source row is done an output row is complete: the epilogue reads the slot, ZEROES it (every MMA
//     accumulates; no first-MMA special case inside a multi-slot instruction) and hands it back, then folds the a_x axis
//     through shared memory exactly like tc_recon_ts.cu (col2im along x) and writes R / the energy partial.
// cfg3: 4 K steps x 3 (hi*hi, lo*hi, hi*lo) MMAs of N = 240 per source row (120 clk each with the operand in tensor
// memory) instead of 180 MMAs of N = 16 per output row; 225 taps x 32 atoms per output cost 1440 tensor-pipe clocks per
// 128-column row against 7200 FMA-pipe clocks.
//
// Roles (576 threads): warps 0-7 write the operand stages (warp w: lane quarter w % 4, atom half w / 4; two rows in
// flight), warp 8 issues the MMAs (ONE issuer: all contributions to a slot are then executed in program order - MMAs of
// different warps are not - so the truncating accumulation stays bitwise reproducible), warp 9 idles, warps 10-17 are two
// epilogue groups serving alternate output rows (RSD is even: a slot always belongs to the same group).
// mbarriers: a_full/a_free per operand stage, d_full/d_free per ring slot.
#include "tc_common.cuh"

namespace tnmf {
namespace tc {
namespace rco {

using tiled::ceil_div;
using tiled::Geo2;
using tiled::round_up;

constexpr int kTile = 128;
constexpr int kEpiGroups = 2;           // epilogue groups of 4 warps: output row g belongs to group g % 2
constexpr int kThreads = 32 * (8 + 2 + 4 * kEpiGroups);
constexpr int kRingMax = 16;            // output-row accumulators
constexpr int kStageMax = 4;            // operand stages
constexpr int kMaxSmem = 226 * 1024;
constexpr int kAtomsPerThread = 16;     // most operand columns one writing thread takes per row (half of the padded atoms)

struct Plan {
    int KM, ksteps;                 // atoms padded to a multiple of 8
    int NU, NP, NB;                 // C * AX, its padding to a multiple of 16, rows of the atom operand = AY * NP
    int VW, S;                      // virtual columns per sample, new output columns per tile
    int RSD, NST, a_col0;           // accumulator slots, operand stages, first TMEM column of the stages
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
    if (g.C < 1 || g.AY < 2 || g.AX < 1 || g.AX > 64) return false;
    p.KM = round_up(g.M, 8);
    if (p.KM > 2 * kAtomsPerThread || (long long)kAtomsPerThread * g.hsm >= (1ll << 31)) return false;
    p.ksteps = p.KM / 8;
    p.NU = g.C * g.AX;
    p.NP = round_up(p.NU, 16);
    if (p.NP > 48 || g.AY * p.NP > 256) return false;      // one MMA covers the whole window
    p.NB = g.AY * p.NP;
    // TMEM: RSD accumulator slots (even, >= AY + 1: the window plus the row being drained), then NST >= 2 operand stages
    p.RSD = round_up(g.AY + 1, 2);
    if (p.RSD > kRingMax || p.RSD * p.NP + 2 * 2 * p.KM > 512) return false;
    while (p.RSD + 2 <= kRingMax && (p.RSD + 2) * p.NP + 3 * 2 * p.KM <= 512) p.RSD += 2;
    p.NST = (512 - p.RSD * p.NP) / (2 * p.KM);
    if (p.NST > kStageMax) p.NST = kStageMax;
    p.a_col0 = p.RSD * p.NP;
    p.VW = g.DX + g.AX - 1;
    p.S = kTile - (g.AX - 1);
    p.b_floats = p.NB * p.KM;
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

// C: channels (compile time: the epilogue's sums live in registers); APT: atoms per stage-writing thread = KM / 2;
// P3: plane mode (G = Geo3, tc_common.cuh) - virtual samples (n, z), H shifted by the host to plane z + offz - az, atom
// plane az of W, and R accumulated over the launches of one reconstruction (g.acc)
template <int C, int APT, bool P3, class G>
__device__ __forceinline__ void recon_os_body(const G &g, const Plan &p, const Args &a) {
    extern __shared__ __align__(128) float smem[];
    __shared__ __align__(8) unsigned long long a_full[kStageMax], a_free[kStageMax], d_full[kRingMax], d_free[kRingMax];
    __shared__ unsigned tmem_base_s;
    const int tid = threadIdx.x, warp = __shfl_sync(0xffffffffu, tid >> 5, 0), lane = tid & 31;
    const int KM = p.KM, AY = g.AY, AX = g.AX, RSD = p.RSD, NST = p.NST, NP = p.NP, NU = p.NU, NB = p.NB;
    float *b_hi = smem, *b_lo = smem + p.b_floats;
    float *psm = b_lo + p.b_floats;                             // [group][2][NP][128]: P of one output row, (c, ax)-major

    if (tid == 0) {
        for (int s = 0; s < kStageMax; ++s) { mbar_init(&a_full[s], 8); mbar_init(&a_free[s], 1); }
        for (int s = 0; s < kRingMax; ++s) { mbar_init(&d_full[s], 1); mbar_init(&d_free[s], 4); }
        mbar_fence_init();
    }
    if (warp == 8) tmem_alloc(&tmem_base_s, 512);
    // atom operand: B[n = ay*NP + c*AX + ax][k = m] = W[m, c, ay, ax]   (zero rows / atoms beyond)
    for (int idx = tid; idx < NB * KM; idx += kThreads) {
        const int n = idx / KM, m = idx - n * KM;
        const int ay = n / NP, r = n - ay * NP;
        float v = 0.f;
        if (r < NU && m < g.M) {
            const int c = r / AX, ax = r - c * AX;
            if constexpr (P3) v = a.W[((((long long)m * C + c) * g.AZ + g.az) * AY + ay) * AX + ax];
            else v = a.W[(((long long)m * C + c) * AY + ay) * AX + ax];
        }
        float hi, lo;
        split_tf32(v, hi, lo);
        const size_t o = canon_offset_floats(n, m, NB);
        b_hi[o] = hi;
        b_lo[o] = lo;
    }
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const unsigned tmem_base = tmem_base_s;
    if (warp < 4) {                                             // every MMA accumulates: the slots start at zero
        for (int c = 0; c < p.a_col0; c += 16) tmem_st16_zero(tmem_base + ((unsigned)(warp * 32) << 16) + (unsigned)c);
        tmem_st_wait();
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();

    if (warp < 8) {
        // ------------------------------------ stage writers ------------------------------------
        const int quarter = warp & 3, half = warp >> 2;
        const int i = quarter * 32 + lane;                      // column of the tile = TMEM lane
        const int m_lo = half * APT;                            // this thread's atoms: [m_lo, m_lo + APT) of the KM padded ones
        const int m_valid = max(0, min(APT, g.M - m_lo));
        const unsigned t_lane = tmem_base + ((unsigned)(quarter * 32) << 16) + (unsigned)(p.a_col0 + m_lo);
        int st = 0;
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
            // two rows are always in flight (the activations come from DRAM: ~1000 clk against ~1500 clk per row)
            long long hbase;
            if constexpr (P3) hbase = (long long)(n / g.NZ) * g.hsn + (long long)(n % g.NZ) * g.hsz;
            else hbase = (long long)n * g.hsn;
            const float *hnext = a.H + (real ? hbase + (long long)m_lo * g.hsm + v + (long long)w.ta * g.hsy : 0);
            const int mv = real ? m_valid : 0;
            float hva[APT], hvb[APT];
            auto load_row = [&](float (&hv)[APT]) {
#pragma unroll
                for (int e = 0; e < APT; ++e) hv[e] = e < mv ? __ldg(hnext + (unsigned)e * (unsigned)g.hsm) : 0.f;
                hnext += g.hsy;
            };
            auto write_row = [&](const float (&hv)[APT]) {
                if (wraps) TC_PROF_WAIT(afree, mbar_wait_backoff(&a_free[st], (wraps - 1u) & 1u, 20));
                tc_fence_after();
                const unsigned t_hi = t_lane + (unsigned)(st * 2 * KM), t_lo = t_hi + (unsigned)KM;
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
                if (lane == 0) mbar_arrive(&a_full[st]);
                if (++st == NST) { st = 0; ++wraps; }
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
        if (blockIdx.x == 0 && tid == 0) printf("recon_os writers: total %lld  wait a_free %lld\n", prof_total, prof_afree);
#endif
    } else if (warp >= 10) {
        // ------------------------------------ epilogue: fold the a_x axis ------------------------------------
        const int q = warp & 3, grp = (warp - 10) >> 2;
        const int i = q * 32 + lane;                            // TMEM lane = column of the tile
        const unsigned lane_base = tmem_base + ((unsigned)(q * 32) << 16);
        const long long plane = (long long)g.DY * g.DX;
        float *psm_g = psm + (size_t)grp * 2 * NP * kTile;
        double e_local = 0.0;
        int slot = 0;
        unsigned slot_wraps = 0, prow = 0, row = 0;             // row: output rows of this CTA so far (all groups)
        TC_PROF_DECL(dfull); TC_PROF_DECL(total);
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
            long long obase, cstride = plane;
            if constexpr (P3) {
                obase = (long long)(n / g.NZ) * g.xsn + (long long)(n % g.NZ) * plane + xo;
                cstride = g.xsc;
            } else {
                obase = (long long)n * C * plane + xo;
            }
            for (int y = w.y0; y < w.y1; ++y, ++row) {
                const int my_slot = slot;
                const unsigned my_par = slot_wraps & 1u;
                if (++slot == RSD) { slot = 0; ++slot_wraps; }
                if ((int)(row % kEpiGroups) != grp) continue;
                float *ps = psm_g + (size_t)(prow & 1u) * NP * kTile;
                ++prow;
                TC_PROF_WAIT(dfull, mbar_wait_backoff(&d_full[my_slot], my_par, 20));
                tc_fence_after();
                // all columns of the row in registers, the slot zeroed and handed back after one TMEM round trip
                float v[3][16];
#pragma unroll
                for (int h = 0; h < 3; ++h)
                    if (16 * h < NP) tmem_ld16(lane_base + (unsigned)(my_slot * NP + 16 * h), v[h]);
                tmem_ld_wait();
#pragma unroll
                for (int h = 0; h < 3; ++h)
                    if (16 * h < NP) tmem_st16_zero(lane_base + (unsigned)(my_slot * NP + 16 * h));
                tmem_st_wait();
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(&d_free[my_slot]);
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
                asm volatile("bar.sync %0, 128;\n" ::"r"(2 + grp) : "memory");
                if (active) {
                    // R[c, y, x] = sum_ax P[(c, ax)][i + AX-1 - ax]; all loads of a batch are issued before the first add
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
                        const long long o = obase + (long long)c * cstride + (long long)y * g.DX;
                        if constexpr (P3) {
                            if (g.acc) r[c] = a.R[o] + r[c];
                        }
                        if (a.R) a.R[o] = r[c];
                        if (a.V) {
                            const double d = (double)a.V[o] - (double)r[c];
                            e_local += d * d;
                        }
                    }
                }
            }
        }
#ifdef TNMF_TC_PROFILE
        prof_total += clock64();
        if (blockIdx.x == 0 && tid == 10 * 32) printf("recon_os epilogue: total %lld  wait d_full %lld\n", prof_total, prof_dfull);
#endif
        if (a.epart) {                                          // one partial per epilogue warp
            for (int o = 16; o > 0; o >>= 1) e_local += __shfl_xor_sync(0xffffffffu, e_local, o);
            if (lane == 0) a.epart[(long long)blockIdx.x * (4 * kEpiGroups) + grp * 4 + q] = e_local;
        }
    } else if (warp == 8) {
        // ------------------------------------ MMA issuer (one converged warp, one elected lane) ------------------------------------
        const unsigned tmem_u = __shfl_sync(0xffffffffu, tmem_base, 0);
        const unsigned desc_hi = (128u >> 4) | (1u << 14);      // SBO = 128, descriptor version 1
        // low descriptor words: start address (>> 4) + LBO field (LBO = NB * 16 bytes); a row offset of n rows (a multiple
        // of 8) advances the start address by n * 16 bytes, a K step by 2 * LBO
        const unsigned w_hi = __shfl_sync(0xffffffffu, (smem_u32(b_hi) >> 4) + ((unsigned)NB << 16), 0);
        const unsigned w_lo = __shfl_sync(0xffffffffu, (smem_u32(b_lo) >> 4) + ((unsigned)NB << 16), 0);
        const unsigned b_step16 = 2u * (unsigned)NB;
        constexpr int kSteps = APT / 4;                         // K steps: KM = 2 * APT atoms, 8 per MMA (compile time: the
        int st = 0;                                             // issue loop is uniform adds between MMAs, nothing else)
        unsigned ph = 0;
        int slot_in = 0, slot_lo = 0, slot_out = 0;            // slot of the next row to enter / of the window's first row /
        unsigned wraps_in = 0;                                  // of the next row to complete
        TC_PROF_DECL(afull); TC_PROF_DECL(dfree); TC_PROF_DECL(total); TC_PROF_DECL(issue);
#ifdef TNMF_TC_PROFILE
        prof_total = -clock64();
#endif
        // The one issuing warp is also the one that keeps the books (which rows enter the window, where it wraps, which
        // stage and which slots to wait for): ~700 clk per source row, during which the pipe ran dry (profiled: 38 % of
        // the kernel).  The loop is therefore SOFTWARE-PIPELINED: the books and the waits of source row i + 1 are done
        // after all but the last K step of row i have been issued - under MMAs that are executing or queued - and only
        // then follow the last K step of row i and its commits.
        // A slot is waited for (d_free) in `prep` only when the row it held was committed before: prep of source row i + 1
        // runs before the commits of row i, and where row i completes many output rows at once (the bottom of a 'full'
        // problem) while row i + 1 opens the next segment with up to A_y rows, the slot can hold a row that row i
        // completes - waiting for it there would never return.  Such waits follow the commits of row i (`wait_late`).
        struct Row {
            bool valid;
            int st, second, done;                               // operand stage, rows past the ring's wrap, rows this row completes
            int n_late, late_slot;                              // entering rows whose slots are waited for after the commits
            unsigned late_wraps;
            unsigned d0, bo, bo1, idesc0, idesc1, ta_hi, ta_lo;
        };
        long long u = blockIdx.x;
        Unit w = make_unit(u, g, p);
        bool in_unit = u < p.units && w.y0 < w.y1;
        int ty = w.ta, next_in = w.y0, win_lo = w.y0, next_out = w.y0;
        long long rows_in = 0, rows_out = 0;                    // output rows of this CTA entered / committed so far
        auto prep = [&]() {
            Row r;
            r.valid = in_unit;
            r.n_late = 0;
            if (!in_unit) return r;
            const int yhi = min(w.y1 - 1, ty - g.offy + AY - 1), ylo = max(w.y0, ty - g.offy);
            // output rows that enter the window with this source row: their slots must have been drained
            for (; next_in <= yhi; ++next_in, ++rows_in) {
                if (wraps_in) {
                    if (rows_in - RSD < rows_out) TC_PROF_WAIT(dfree, mbar_wait(&d_free[slot_in], (wraps_in - 1u) & 1u));
                    else if (r.n_late++ == 0) { r.late_slot = slot_in; r.late_wraps = wraps_in; }
                }
                if (++slot_in == RSD) { slot_in = 0; ++wraps_in; }
            }
            for (; win_lo < ylo; ++win_lo)
                if (++slot_lo == RSD) slot_lo = 0;
            TC_PROF_WAIT(afull, mbar_wait(&a_full[st], ph));
            tc_fence_after();
            const int cnt = yhi - ylo + 1;                      // >= 1: every source row of a unit meets one of its output rows
            const int first = min(cnt, RSD - slot_lo);
            r.second = cnt - first;
            r.bo = (unsigned)((ylo + g.offy - ty) * NP);        // first row block of B: ay of the window's first row
            r.bo1 = r.bo + (unsigned)(first * NP);
            r.d0 = tmem_u + (unsigned)(slot_lo * NP);
            r.idesc0 = idesc_tf32(kTile, first * NP);
            r.idesc1 = idesc_tf32(kTile, max(r.second, 1) * NP);
            r.ta_hi = tmem_u + (unsigned)(p.a_col0 + st * 2 * KM);
            r.ta_lo = r.ta_hi + (unsigned)KM;
            r.st = st;
            if (++st == NST) { st = 0; ph ^= 1u; }
            // output rows whose last source row this is (at the bottom of a 'full' problem several at once)
            const int done_to = ty == w.tb ? w.y1 : min(w.y1, ty - g.offy + 1);
            r.done = max(done_to - next_out, 0);
            next_out += r.done;
            // advance to the next source row (of the next segment when this one is finished)
            if (++ty > w.tb) {
                u += gridDim.x;
                in_unit = u < p.units;
                if (in_unit) {
                    w = make_unit(u, g, p);
                    in_unit = w.y0 < w.y1;
                    ty = w.ta; next_in = w.y0; win_lo = w.y0; next_out = w.y0;
                    slot_lo = slot_in;                          // the segment's first output row enters here
                }
            }
            return r;
        };
        auto issue = [&](const Row &r, int ks_a, int ks_b) {     // K steps [ks_a, ks_b) of a row (compile-time bounds when inlined)
            if (r.second > 0) {                                 // the window wraps around the ring: two runs of slots
#pragma unroll
                for (int ks = 0; ks < kSteps; ++ks)
                    if (ks >= ks_a && ks < ks_b) {
                        const unsigned kb = r.bo + (unsigned)ks * b_step16, kb1 = r.bo1 + (unsigned)ks * b_step16;
                        mma_tf32_ts2<true>(r.d0, r.ta_hi + 8u * ks, w_hi + kb, desc_hi, r.idesc0);
                        mma_tf32_ts2<true>(tmem_u, r.ta_hi + 8u * ks, w_hi + kb1, desc_hi, r.idesc1);
                        mma_tf32_ts2<true>(r.d0, r.ta_lo + 8u * ks, w_hi + kb, desc_hi, r.idesc0);
                        mma_tf32_ts2<true>(tmem_u, r.ta_lo + 8u * ks, w_hi + kb1, desc_hi, r.idesc1);
                        mma_tf32_ts2<true>(r.d0, r.ta_hi + 8u * ks, w_lo + kb, desc_hi, r.idesc0);
                        mma_tf32_ts2<true>(tmem_u, r.ta_hi + 8u * ks, w_lo + kb1, desc_hi, r.idesc1);
                    }
            } else {
#pragma unroll
                for (int ks = 0; ks < kSteps; ++ks)
                    if (ks >= ks_a && ks < ks_b) {
                        const unsigned kb = r.bo + (unsigned)ks * b_step16;
                        mma_tf32_ts2<true>(r.d0, r.ta_hi + 8u * ks, w_hi + kb, desc_hi, r.idesc0);
                        mma_tf32_ts2<true>(r.d0, r.ta_lo + 8u * ks, w_hi + kb, desc_hi, r.idesc0);
                        mma_tf32_ts2<true>(r.d0, r.ta_hi + 8u * ks, w_lo + kb, desc_hi, r.idesc0);
                    }
            }
        };
        auto wait_late = [&](const Row &r) {
            if (!r.n_late) return;
            int s = r.late_slot;
            unsigned wr = r.late_wraps;
            for (int i = 0; i < r.n_late; ++i) {
                TC_PROF_WAIT(dfree, mbar_wait(&d_free[s], (wr - 1u) & 1u));
                if (++s == RSD) { s = 0; ++wr; }
            }
            tc_fence_after();
        };
        Row cur = prep();
        wait_late(cur);
        while (cur.valid) {
#ifdef TNMF_TC_PROFILE
            const long long t_i = clock64();
#endif
            if (kSteps > 1 && elect_one()) issue(cur, 0, kSteps - 1);
            __syncwarp();
#ifdef TNMF_TC_PROFILE
            prof_issue += clock64() - t_i;
#endif
            const Row nxt = prep();
#ifdef TNMF_TC_PROFILE
            const long long t_j = clock64();
#endif
            if (elect_one()) issue(cur, kSteps > 1 ? kSteps - 1 : 0, kSteps);
            __syncwarp();
#ifdef TNMF_TC_PROFILE
            prof_issue += clock64() - t_j;
#endif
            mma_commit_elect(&a_free[cur.st]);
            for (int i = 0; i < cur.done; ++i) {
                mma_commit_elect(&d_full[slot_out]);
                if (++slot_out == RSD) slot_out = 0;
            }
            rows_out += cur.done;
            wait_late(nxt);
            cur = nxt;
        }
#ifdef TNMF_TC_PROFILE
        prof_total += clock64();
        if (blockIdx.x == 0 && lane == 0)
            printf("recon_os mma: total %lld  wait a_full %lld  wait d_free %lld  issuing %lld\n", prof_total, prof_afull, prof_dfree, prof_issue);
#endif
        __syncwarp();
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 8) tmem_dealloc(tmem_base, 512);
}

template <int C, int APT>
__global__ void __launch_bounds__(kThreads, 1) recon_os_kernel(const Geo2 g, const Plan p, const Args a) {
    recon_os_body<C, APT, false>(g, p, a);
}
template <int C, int APT>
__global__ void __launch_bounds__(kThreads, 1) recon_os3_kernel(const Geo3 g, const Plan p, const Args a) {
    recon_os_body<C, APT, true>(g, p, a);
}
template <int C, int APT> static auto kernel_for(const Geo2 &) { return recon_os_kernel<C, APT>; }
template <int C, int APT> static auto kernel_for(const Geo3 &) { return recon_os3_kernel<C, APT>; }

template <int C, int APT, class G>
static int launch2(const G &g, const Plan &p, const Args &a, cudaStream_t st) {
    auto kern = kernel_for<C, APT>(g);
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, kMaxSmem);
    if (e != cudaSuccess) return status_from_cuda(e);
    kern<<<(unsigned)p.grid, kThreads, p.smem, st>>>(g, p, a);
    TNMF_CHECK_LAUNCH();
    return TNMF_OK;
}

template <int C, class G>
static int launch(const G &g, const Plan &p, const Args &a, cudaStream_t st) {
    switch (p.KM / 2) {
        case 4: return launch2<C, 4>(g, p, a, st);
        case 8: return launch2<C, 8>(g, p, a, st);
        case 12: return launch2<C, 12>(g, p, a, st);
        case 16: return launch2<C, 16>(g, p, a, st);
        default: return TNMF_EUNSUPPORTED;
    }
}

}  // namespace rco
}  // namespace tc

// ---- dispatch ----------------------------------------------------------------------------------------------------------
bool tc_recon_os_supported(const Geo &g, int dtype) {
    tc::rco::Plan p;
    if (plane_problem(g))
        return g.C <= 2 && tc::plane_mode_ok(g, dtype) && tc::rco::make_plan(tc::make_geo3(g, false), p);
    if (!tc::rank2_ok(g, dtype) || g.C > 2) return false;
    return tc::rco::make_plan(tiled::make_geo2(g), p);
}

int tc_recon_os_partials(const Geo &g) {
    tc::rco::Plan p;
    const bool ok = plane_problem(g) ? tc::rco::make_plan(tc::make_geo3(g, false), p)
                                         : tc::rco::make_plan(tiled::make_geo2(g), p);
    return ok ? p.grid * 4 * tc::rco::kEpiGroups : 0;
}

template <class G>
static int reconstruct_os(const G &q, const Geo &g, const tc::rco::Plan &p, const tc::rco::Args &a, cudaStream_t st) {
    switch (g.C) {
        case 1: return tc::rco::launch<1>(q, p, a, st);
        case 2: return tc::rco::launch<2>(q, p, a, st);
        default: return TNMF_EUNSUPPORTED;
    }
}

int tc_reconstruct_os(const Geo &g, const float *W, const float *H, float *R, const float *V, double *energy_partials,
                      int *n_partials, cudaStream_t st) {
    const bool planes = plane_problem(g);
    tc::Geo3 q3 = tc::make_geo3(g, false);
    const tiled::Geo2 q = planes ? q3 : tiled::make_geo2(g);
    tc::rco::Plan p;
    if (!tc::rco::make_plan(q, p)) return TNMF_EUNSUPPORTED;
    tc::rco::Args a;
    a.W = W; a.H = H; a.V = V; a.R = R; a.epart = energy_partials;
    if (n_partials) *n_partials = p.grid * 4 * tc::rco::kEpiGroups;
    if (!planes) return reconstruct_os(q, g, p, a, st);
    // 3-D: one launch per atom plane a_z, in order - the first writes R, the others add to it (deterministic); the last
    // one holds the complete R and computes the energy partials
    if (!R) return TNMF_EINVAL;
    for (int az = 0; az < g.A[0]; ++az) {
        q3.az = az;
        q3.acc = az > 0;
        a.H = H + (long long)(q3.offz - az) * q3.hsz;
        a.V = az + 1 == g.A[0] ? V : nullptr;
        a.epart = az + 1 == g.A[0] ? energy_partials : nullptr;
        const int s = reconstruct_os(q3, g, p, a, st);
        if (s) return s;
    }
    return TNMF_OK;
}

int tc_recon_os_launches(const Geo &g) { return g.A[0]; }

}  // namespace tnmf
