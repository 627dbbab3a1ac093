// Tensor-core (tcgen05, 3xTF32) W gradient for NARROW atoms (C * A_x <= 16): hi / lo halves, two source rows and both tensors
// STACKED IN THE MMA LANES, expanded operand in tensor memory.
//
//   neg[m,c,ay,ax] = sum_n sum_{ty,tx} H[n,m,ty,tx] * Vext[n,c,ty-offy+ay,tx-offx+ax]      (tnmf/backends/NumPy.py:77-85)
//   pos[m,c,ay,ax] = the same with R                                                       (tnmf/backends/NumPy.py:80,87-90)
//
// tc_gradw_ts.cu puts the taps (X, c, ax) of ONE source row into the 128 MMA lanes and pays three MMAs per product
// (hi*hi, lo*hi, hi*lo).  With C * A_x = 15 (BASELINE config 3) that is 30 of 128 lanes.  Here a lane is
//       L = part * 64 + s * 32 + X * 16 + k        part: hi / lo half of the split,  s: source row r or r + 1,
//                                                  X: V or R,  k = c * A_x + ax  (< 16)
// so ALL lanes carry taps and the hi/lo split of the expanded operand costs lanes instead of instructions:
//       D'[L, (j, m)] += sum_col A'[L, col] * Bhi[(j, m), col]      and      += ... * Blo[(j, m), col]
// are the only two MMAs per K step (the second one adds hi*lo - and lo*lo, which the 3xTF32 scheme merely drops).  The four
// (part, s) groups are separate per-CTA partial slices that finish_gradient_w adds in its fixed-order double sum.
//   * B' = ring of activation rows [(slot, atom), column] in shared memory, hi and lo copies, 8 atoms per launch; window
//     position j of a step is the activation row t = r + offy - A_y + 1 + j; lane group s pairs it with atom row
//     ay = A_y - 1 - j + s (entries with ay outside [0, A_y) are computed and never read).
//   * the window ALWAYS has WP = roundup(A_y + 1, 4) positions: activation rows outside the unit's band [ty0, ty1) are staged
//     as rows of zeros, so every MMA has the same N = 8 * WP / 2 (a multiple of 16) and no clipping logic exists;
//   * a step = two source rows; the first WP - 1 ring slots are mirrored behind the last, so a window is one run of slots.
// Everything else follows tc_gradw_ts.cu: the accumulator lives in TMEM in two sets that alternate every kEpochSteps steps
// (the tensor core truncates when it adds: chains are cut), four drainer warps add a finished set into the CTA's slices and
// zero it, two issuing warps own a STATIC half of the window positions each (a TMEM column is written by one warp only: the
// accumulation order is fixed, results are bitwise reproducible), workers expand straight from a raw-row buffer into TMEM.
// cfg3 (32 atoms of 15 x 15, one channel): 2 MMAs of N = 64 per issuer and K step for 2 source rows x 8 atoms, against
// 3 MMAs of N = 256 for 2 source rows x 16 atoms in tc_gradw.cu - two thirds of the tensor-pipe time.
#include "tc_common.cuh"

namespace tnmf {
namespace tc {
namespace gwn {

using tiled::ceil_div;
using tiled::Geo2;
using tiled::round_up;

constexpr int kCT = 64;             // activation columns per tile
constexpr int kNB = 8;              // atoms per launch
constexpr int kKS = 64;             // tile columns per operand stage = the whole tile: one stage per step
constexpr int kWorkers = 256;
constexpr int kIssuers = 4;          // issuing warps (two when the window does not split four ways)
constexpr int kThreads = 32 * (8 + kIssuers + 4);
constexpr int kEpochSteps = 12;     // steps (two source rows each) accumulated into one TMEM set before it is drained:
                                    // 12 x 8 K steps x 2 = 192 additions per accumulator, the chain length of tc_gradw_ts.cu
constexpr int kMaxAStages = 4;
constexpr int kRingMax = 32;
constexpr int kRawMax = 4;          // raw elements per worker and step: 4 * C * (64 + AX - 1) <= 1024
constexpr int kMaxSmem = 226 * 1024;

struct Plan {
    int KPL;                        // taps per tensor and source row = C * AX (<= 16)
    int TXP, RW, RWp, rawX, raw_floats, nraw;
    int WP, NA, n_astages, a_col0;  // window positions, accumulator columns per set, operand stages, their first column
    int n_issue;                    // issuing warps in use: 4 when WP is a multiple of 8 (N = 2 * WP per MMA), else 2
    int RS, NRr, ring_floats;       // logical ring slots (even), physical ring rows = (RS + WP - 1) * 8, floats of one half
    int tiles;
    long long total, quota, units;
    int grid;
    size_t smem;
};

struct Args {
    const float *V, *R, *H;
    float *partials;                // [grid * 4][2][M*C*AY*AX]
    int m0;
};

// max_grid > 0: at most that many CTAs (longer ranges per CTA), so that the partial slices fit a workspace planned
// for a larger problem
bool make_plan(const Geo2 &g, Plan &p, int max_grid = 0) {
    p = Plan();
    if (g.AY < 1 || g.AY > 19) return false;
    p.KPL = g.C * g.AX;
    if (p.KPL > 16) return false;
    p.WP = round_up(g.AY + 1, 4);
    p.NA = kNB * p.WP;
#ifndef TNMF_GWN_MAX_ISSUERS
#define TNMF_GWN_MAX_ISSUERS 2
#endif
    p.n_issue = (p.WP % 8 == 0 && TNMF_GWN_MAX_ISSUERS >= 4) ? 4 : 2;
    p.n_astages = (512 - 2 * p.NA) / kKS;
    if (p.n_astages < 2) return false;
    if (p.n_astages > kMaxAStages) p.n_astages = kMaxAStages;
    p.a_col0 = 2 * p.NA;
    p.TXP = g.TX + g.AX - 1;
    p.RW = kCT + g.AX - 1;
    // channel pitch == AX (mod 32) and plane pitch == 16 (mod 32): lane (X, k = (c, ax)) of a warp then reads word
    // X * rawX + c * RWp + ax + col == 16 X + k + col (mod 32): no bank conflicts
    p.RWp = p.RW + 1;
    while ((p.RWp - g.AX) % 32 != 0) ++p.RWp;
    p.rawX = g.C * p.RWp;
    while (p.rawX % 32 != 16) ++p.rawX;
    p.raw_floats = 4 * p.rawX + 128;                        // planes (s, X), zeros for the idle lanes
    p.nraw = ceil_div(4 * g.C * p.RW, kWorkers);
    if (p.nraw > kRawMax) return false;
    const size_t fixed = (size_t)2 * p.raw_floats * 4 + 1024;
    for (p.RS = kRingMax; p.RS >= p.WP + 4; p.RS -= 2) {
        p.NRr = (p.RS + p.WP - 1) * kNB;
        p.ring_floats = (p.NRr * 4 + 4) * (kCT / 4);        // K-chunk stride padded by 16 bytes: conflict-free row staging
        if (fixed + (size_t)2 * p.ring_floats * 4 <= (size_t)kMaxSmem) break;
    }
    if (p.RS < p.WP + 4) return false;
    p.smem = fixed + (size_t)2 * p.ring_floats * 4;
    const long long cols = (long long)g.N * p.TXP;
    if (cols <= 0 || cols >= (1ll << 31) - kCT) return false;
    p.tiles = (int)((cols + kCT - 1) / kCT);
    const int sms = tma::sm_count();
    p.total = (long long)p.tiles * g.TY;                    // equal linear ranges of the (tile, row) space, one per CTA
    p.quota = (p.total + sms - 1) / sms;
    const long long min_quota = g.TY < 8 ? g.TY : 8;
    if (p.quota < min_quota) p.quota = min_quota;
    if (max_grid > 0 && (p.total + p.quota - 1) / p.quota > max_grid) p.quota = (p.total + max_grid - 1) / max_grid;
    p.grid = (int)((p.total + p.quota - 1) / p.quota);
    p.units = (long long)p.grid * ((p.quota + g.TY - 2) / g.TY + 1);
    return true;
}

struct Unit {
    int tile, ty0, ty1, r_lo, steps, j00;   // activation rows [ty0, ty1), first source row, steps, window base of step 0
};
__device__ __forceinline__ Unit make_unit(long long u, const Geo2 &g, const Plan &p) {
    Unit w;
    const long long b = u % p.grid, k = u / p.grid;
    const long long lo = b * p.quota, hi = min(lo + p.quota, p.total);
    w.tile = (int)(lo / g.TY + k);
    const long long t0 = (long long)w.tile * g.TY;
    const long long s0 = max(lo, t0), s1 = min(hi, t0 + g.TY);
    w.ty0 = s1 > s0 ? (int)(s0 - t0) : 0;
    w.ty1 = s1 > s0 ? (int)(s1 - t0) : 0;
    w.r_lo = max(0, w.ty0 - g.offy);
    const int r_hi = min(g.DY - 1, w.ty1 - 1 - g.offy + g.AY - 1);
    w.steps = (r_hi - w.r_lo + 2) / 2;
    w.j00 = w.r_lo + g.offy - g.AY + 1;
    return w;
}

// P3: plane mode (G = Geo3, tc_common.cuh) - virtual samples (n, z), H shifted by the host to plane z + offz - az, the
// partial slices indexed [m][c][a_z][a_y][a_x] with this launch's a_z
template <bool P3, class G>
__device__ __forceinline__ void gradw_ns_body(const G &g, const Plan &p, const Args &a) {
    extern __shared__ __align__(128) float smem[];
    __shared__ __align__(8) unsigned long long a_full[kMaxAStages], a_empty[kMaxAStages], h_full[kRingMax / 2], h_free[kRingMax / 2],
        set_done[2], set_free[2];
    __shared__ unsigned tmem_base_s;
    const int tid = threadIdx.x, warp = __shfl_sync(0xffffffffu, tid >> 5, 0), lane = tid & 31;
    const int AY = g.AY, AX = g.AX, C = g.C, RS = p.RS, RW = p.RW, WP = p.WP;
    float *ring_hi = smem, *ring_lo = smem + p.ring_floats;
    float *raw = ring_lo + p.ring_floats;                       // [2 buffers][plane (s, X)][rawX] + zeros

    if (tid == 0) {
        // (h_full / h_free guard PAIRS of ring slots: activation rows enter and leave two at a time)
        for (int s = 0; s < kMaxAStages; ++s) { mbar_init(&a_full[s], 8); mbar_init(&a_empty[s], p.n_issue); }
        for (int s = 0; s < kRingMax / 2; ++s) { mbar_init(&h_full[s], kWorkers); mbar_init(&h_free[s], p.n_issue); }
        for (int s = 0; s < 2; ++s) { mbar_init(&set_done[s], p.n_issue); mbar_init(&set_free[s], 128); }
        mbar_fence_init();
    }
    if (warp == 8) tmem_alloc(&tmem_base_s, 512);
    for (int idx = tid; idx < 2 * p.raw_floats; idx += kThreads) raw[idx] = 0.f;     // pads and the idle lanes' zeros
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const unsigned tmem_base = tmem_base_s;
    if (warp < 4) {                                             // accumulators = 0, idle operand lanes = 0
        for (int c = 0; c < 512; c += 16) tmem_st16_zero(tmem_base + ((unsigned)(warp * 32) << 16) + (unsigned)c);
        tmem_st_wait();
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();

    long long count = (long long)g.M * C * AY * AX;
    if constexpr (P3) count *= g.AZ;

    if (warp < 8) {
        // ------------------------------------ workers ------------------------------------
        const int quarter = warp & 3, half = warp >> 2;
        const int L = quarter * 32 + lane;                      // operand lane of this thread
        const int part = L >> 6, s_l = (L >> 5) & 1, X_l = (L >> 4) & 1, k = L & 15;
        const bool live = k < p.KPL;
        // idle lanes (k >= C * AX, so k = 15 is one of them) read zeros from bank 15 + col, which no live lane of the warp uses
        const int src_off = live ? (s_l * 2 + X_l) * p.rawX + (k / AX) * p.RWp + (k % AX) : 4 * p.rawX + 15;
        const unsigned t_lane = tmem_base + ((unsigned)(quarter * 32) << 16) + (unsigned)(p.a_col0 + half * (kKS / 2));   // 32 columns
        int st = 0;
        unsigned a_wraps = 0, buf = 0;
        const long long plane = (long long)g.DY * g.DX;
        const int raw_count = 4 * C * RW;
        const int h_sel = tid >> 7, h_ml = (tid >> 4) & 7, h_cg = tid & 15;     // activation chunk: row of the pair, atom,
        int slot_new = 0;                                                      // columns 4 cg .. 4 cg + 3
        unsigned wraps = 0;
        TC_PROF_DECL(empty); TC_PROF_DECL(hfree); TC_PROF_DECL(bar); TC_PROF_DECL(total); TC_PROF_DECL(stw);
#ifdef TNMF_TC_PROFILE
        prof_total = -clock64();
#endif
        for (long long u = blockIdx.x; u < p.units; u += gridDim.x) {
            const Unit w = make_unit(u, g, p);
            if (w.ty0 >= w.ty1) break;                          // past this CTA's last segment
            const int r_hi = w.r_lo + 2 * w.steps - 1;          // (may be one past the last real row: staged as zeros)
            const int r_last = min(g.DY - 1, w.ty1 - 1 - g.offy + AY - 1);
            // raw slot q = tid + 256 e -> (s, X, c, position): source offset in row r + s (relative to row 0), or -1
            long long roff[kRawMax];
            int rdst[kRawMax], rsx[kRawMax];
#pragma unroll
            for (int e = 0; e < kRawMax; ++e) {
                roff[e] = -1;
                rdst[e] = -1;
                rsx[e] = 0;
                const int q = tid + kWorkers * e;
                if (e < p.nraw && q < raw_count) {
                    const int sx = q / (C * RW), qq = q - sx * (C * RW);    // sx = s * 2 + X
                    const int c = qq / RW, xr = qq - c * RW;
                    rdst[e] = sx * p.rawX + c * p.RWp + xr;
                    rsx[e] = sx;
                    const long long J = (long long)w.tile * kCT + xr;
                    const int n = (int)(J / p.TXP);
                    const int x = (int)(J - (long long)n * p.TXP) - g.offx;
                    if (n < g.N && (unsigned)x < (unsigned)g.DX) {
                        if constexpr (P3) roff[e] = (n / g.NZ) * g.xsn + c * g.xsc + (long long)(g.z0 + n % g.NZ) * plane + x;
                        else roff[e] = ((long long)n * C + c) * plane + x;
                    }
                }
            }
            long long hoff[4];
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const long long J = (long long)w.tile * kCT + 4 * h_cg + e;
                const int n = (int)(J / p.TXP);
                const int xv = (int)(J - (long long)n * p.TXP);
                long long hbase;
                if constexpr (P3) hbase = (long long)(n / g.NZ) * g.hsn + (long long)(g.z0 + n % g.NZ) * g.hsz;
                else hbase = (long long)n * g.hsn;
                hoff[e] = (n < g.N && xv < g.TX && a.m0 + h_ml < g.M) ? hbase + (long long)(a.m0 + h_ml) * g.hsm + xv : -1;
            }
            auto load_raw = [&](int r, float (&rv)[kRawMax]) {
#pragma unroll
                for (int e = 0; e < kRawMax; ++e) {
                    const int row = r + (rsx[e] >> 1);
                    const float *src = (rsx[e] & 1) ? a.R : a.V;
                    rv[e] = (roff[e] >= 0 && row <= r_last) ? __ldg(src + (long long)row * g.DX + roff[e]) : 0.f;
                }
            };
            auto load_h = [&](int t) {                          // this thread's chunk of activation row t (zeros outside the band)
                float4 hv = make_float4(0.f, 0.f, 0.f, 0.f);
                if (t >= w.ty0 && t < w.ty1) {
                    const long long o = (long long)t * g.hsy;
                    hv.x = hoff[0] >= 0 ? a.H[hoff[0] + o] : 0.f;
                    hv.y = hoff[1] >= 0 ? a.H[hoff[1] + o] : 0.f;
                    hv.z = hoff[2] >= 0 ? a.H[hoff[2] + o] : 0.f;
                    hv.w = hoff[3] >= 0 ? a.H[hoff[3] + o] : 0.f;
                }
                return hv;
            };
            auto stage_pair = [&](const float4 &hv) {               // this thread's row of the next pair -> slots slot_new, slot_new + 1
                if (wraps) TC_PROF_WAIT(hfree, mbar_wait_backoff(&h_free[slot_new >> 1], (wraps - 1u) & 1u, 40));
                const int slot = slot_new + h_sel;
                float4 hi, lo;
                split_tf32(hv.x, hi.x, lo.x); split_tf32(hv.y, hi.y, lo.y);
                split_tf32(hv.z, hi.z, lo.z); split_tf32(hv.w, hi.w, lo.w);
                const size_t o = (size_t)slot * 32 + (size_t)h_cg * (p.NRr * 4 + 4) + (size_t)h_ml * 4;
                *reinterpret_cast<float4 *>(ring_hi + o) = hi;
                *reinterpret_cast<float4 *>(ring_lo + o) = lo;
                if (slot < WP - 1) {                                // mirror: a window never wraps
                    const size_t om = o + (size_t)RS * 32;
                    *reinterpret_cast<float4 *>(ring_hi + om) = hi;
                    *reinterpret_cast<float4 *>(ring_lo + om) = lo;
                }
                fence_proxy_async();
                mbar_arrive(&h_full[slot_new >> 1]);
                slot_new += 2;
                if (slot_new == RS) { slot_new = 0; ++wraps; }
            };
            // One step.  Its raw rows and its (last) pair of activation rows were fetched TWO steps ago into (rv, hv): a step
            // lasts ~1000 clk, a DRAM round trip about as long, so a distance of one step left the workers waiting for
            // memory every step.  Once consumed the registers take the loads of step q + 2.
            auto do_step = [&](int q, float (&rv)[kRawMax], float4 &hv) {
                const int r = w.r_lo + 2 * q;
                if (q == 0) {                                       // the whole first window: WP / 2 pairs, the first one prefetched
                    stage_pair(hv);
                    for (int t = w.j00 + 2; t < w.j00 + WP; t += 2) stage_pair(load_h(t + h_sel));
                } else {
                    stage_pair(hv);                                 // rows j00 + WP + 2 (q - 1), + 1
                }
                float *rb = raw + (size_t)buf * p.raw_floats;
#pragma unroll
                for (int e = 0; e < kRawMax; ++e)
                    if (rdst[e] >= 0) rb[rdst[e]] = rv[e];
                if (q + 2 < w.steps) {
                    load_raw(r + 4, rv);
                    hv = load_h(w.j00 + WP + 2 * (q + 1) + h_sel);
                }
                TC_PROF_WAIT(bar, asm volatile("bar.sync 1, 256;\n" ::: "memory"));
                // ---- expansion into tensor memory: lane (part, s, X, c, ax) <- hi or lo of raw[s][X][c][ax + col] ----
                const float *src = rb + src_off + half * (kKS / 2);
                if (a_wraps) TC_PROF_WAIT(empty, mbar_wait_backoff(&a_empty[st], (a_wraps - 1u) & 1u, 20));
                tc_fence_after();
                // hi = the nearest TF32 (add half an ulp of the 10-bit mantissa to the magnitude, clear the low 13 bits: what
                // cvt.rna.tf32 does, without its inf/nan guard - two integer instructions), lo = x - hi (exact).  `part` is
                // uniform in a warp: hi warps never compute lo.
#pragma unroll
                for (int h = 0; h < kKS / 32; ++h) {
                    float v[16];
                    if (part == 0) {
#pragma unroll
                        for (int j = 0; j < 16; ++j)
                            v[j] = __uint_as_float((__float_as_uint(src[h * 16 + j]) + 0x1000u) & 0xffffe000u);
                    } else {
#pragma unroll
                        for (int j = 0; j < 16; ++j) {
                            const float x = src[h * 16 + j];
                            v[j] = x - __uint_as_float((__float_as_uint(x) + 0x1000u) & 0xffffe000u);
                        }
                    }
                    tmem_st16(t_lane + (unsigned)(st * kKS + h * 16), v);
                }
                TC_PROF_WAIT(stw, tmem_st_wait());
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(&a_full[st]);
                if (++st == p.n_astages) { st = 0; ++a_wraps; }
                buf ^= 1u;
            };
            float rva[kRawMax], rvb[kRawMax];
            float4 hva = load_h(w.j00 + h_sel), hvb = make_float4(0.f, 0.f, 0.f, 0.f);
            load_raw(w.r_lo, rva);
            if (w.steps > 1) {
                load_raw(w.r_lo + 2, rvb);
                hvb = load_h(w.j00 + WP + h_sel);
            }
            for (int q = 0; q < w.steps; q += 2) {
                do_step(q, rva, hva);
                if (q + 1 < w.steps) do_step(q + 1, rvb, hvb);
            }
            (void)r_hi;
        }
#ifdef TNMF_TC_PROFILE
        prof_total += clock64();
        if (blockIdx.x == 0 && tid == 0)
            printf("gradw_ns workers: total %lld  wait a_empty %lld  wait h_free %lld  raw barrier %lld  tmem st wait %lld\n", prof_total, prof_empty, prof_hfree, prof_bar, prof_stw);
#endif
    } else if (warp >= 8 + kIssuers) {
        // ------------------------------------ accumulator drainers ------------------------------------
        long long steps_total = 0;
        for (long long u = blockIdx.x; u < p.units; u += gridDim.x) {
            const Unit w = make_unit(u, g, p);
            if (w.ty0 >= w.ty1) break;
            steps_total += w.steps;
        }
        const int n_epochs = (int)((steps_total + kEpochSteps - 1) / kEpochSteps);
        const int l = (warp & 3) * 32 + lane;
        const int part = l >> 6, s_l = (l >> 5) & 1, X_l = (l >> 4) & 1, k = l & 15;
        const bool live = k < p.KPL;
        const int c = live ? k / AX : 0, ax = live ? k - c * AX : 0;
        float *slice = a.partials + ((long long)blockIdx.x * 4 + part * 2 + s_l) * 2 * count + (long long)X_l * count;
        long long mstride = (long long)C * AY * AX;
        float *dst_base = slice + (((long long)a.m0 * C + c) * AY) * AX + ax;
        if constexpr (P3) {
            mstride *= g.AZ;
            dst_base = slice + ((((long long)a.m0 * C + c) * g.AZ + g.az) * AY) * AX + ax;
        }
        TC_PROF_DECL(done); TC_PROF_DECL(total);
#ifdef TNMF_TC_PROFILE
        prof_total = -clock64();
#endif
        for (int e = 0; e < n_epochs; ++e) {
            const int set = e & 1;
            const unsigned tbase = tmem_base + ((unsigned)((warp & 3) * 32) << 16) + (unsigned)(set * p.NA);
            TC_PROF_WAIT(done, mbar_wait_backoff(&set_done[set], (unsigned)((e >> 1) & 1), 100));
            tc_fence_after();
            for (int j = 0; j < WP; ++j) {
                const int ay = AY - 1 - j + s_l;
                float v[8];
                tmem_ld8(tbase + (unsigned)(j * kNB), v);
                tmem_ld_wait();
                tmem_st8_zero(tbase + (unsigned)(j * kNB));
                if (live && ay >= 0 && ay < AY) {
                    float *dst0 = dst_base + (long long)ay * AX;
                    // The slice entry belongs to this thread alone: the first epoch stores, later ones add with a
                    // fire-and-forget reduction (RED.ADD.F32, round to nearest, applied in this thread's program order) -
                    // no dependent load per window position (a read-modify-write cost an L2 round trip for each of them)
#pragma unroll
                    for (int ml = 0; ml < kNB; ++ml)
                        if (a.m0 + ml < g.M) {
                            if (e) atomicAdd(dst0 + ml * mstride, v[ml]);
                            else __stcg(dst0 + ml * mstride, v[ml]);
                        }
                }
            }
            tmem_st_wait();
            tc_fence_before();
            mbar_arrive(&set_free[set]);
        }
#ifdef TNMF_TC_PROFILE
        prof_total += clock64();
        if (blockIdx.x == 0 && tid == 32 * (8 + kIssuers))
            printf("gradw_ns drainers: total %lld  wait set_done %lld  (%d epochs)\n", prof_total, prof_done, n_epochs);
#endif
    } else {
        // ------------------------------------ MMA issuers (converged warps, one elected lane) ------------------------------------
        const unsigned tmem_u = __shfl_sync(0xffffffffu, tmem_base, 0);
        const unsigned lbo_b = (unsigned)p.NRr * 16 + 16;       // ring chunks carry a 16-byte pad
        const unsigned desc_hi = (128u >> 4) | (1u << 14);      // SBO, descriptor version 1
        const unsigned b_lo_word = ((lbo_b >> 4) << 16);
        const unsigned ring_hi16 = __shfl_sync(0xffffffffu, smem_u32(ring_hi) >> 4, 0);
        const unsigned ring_lo16 = __shfl_sync(0xffffffffu, smem_u32(ring_lo) >> 4, 0);
        const unsigned b_step16 = (2 * lbo_b) >> 4;
        // warp X owns the window positions [X * WP / 2, (X + 1) * WP / 2): a TMEM column is written by one warp, in program order
        const int X = warp - 8;
        const int half_w = WP / p.n_issue;                      // window positions of one issuing warp
        const unsigned idesc = idesc_tf32(128, kNB * half_w);
        int st = 0;
        unsigned ph = 0;
        long long steps_done = 0;
        int slot_in = 0, slot_a = 0, slot_out = 0;              // next slot to be filled / first slot of the window / next to free
        unsigned par_in = 0;
        TC_PROF_DECL(full); TC_PROF_DECL(hfull); TC_PROF_DECL(setfree); TC_PROF_DECL(total); TC_PROF_DECL(issue);
#ifdef TNMF_TC_PROFILE
        prof_total = -clock64();
#endif
        for (long long u = blockIdx.x; X < p.n_issue && u < p.units; u += gridDim.x) {
            const Unit w = make_unit(u, g, p);
            if (w.ty0 >= w.ty1) break;
            slot_a = slot_in;                                   // the unit's first window starts where its first row enters
            for (int q = 0; q < w.steps; ++q) {
                const long long epoch = steps_done / kEpochSteps;
                if (steps_done % kEpochSteps == 0 && epoch >= 2) {
                    TC_PROF_WAIT(setfree, mbar_wait(&set_free[epoch & 1], (unsigned)(((epoch >> 1) - 1) & 1)));
                    tc_fence_after();
                }
                const unsigned tset = tmem_u + (unsigned)((epoch & 1) * p.NA) + (unsigned)(X * half_w * kNB);
                // rows that enter the ring with this step: WP at the unit's first step, two afterwards
                for (int i = q ? 2 : WP; i > 0; i -= 2) {
                    TC_PROF_WAIT(hfull, mbar_wait_backoff(&h_full[slot_in >> 1], par_in, 20));
                    slot_in += 2;
                    if (slot_in == RS) { slot_in = 0; par_in ^= 1u; }
                }
                const unsigned b0 = (unsigned)(slot_a + X * half_w) * 8u;       // 8 ring rows = 128 bytes per slot
                TC_PROF_WAIT(full, mbar_wait_backoff(&a_full[st], ph, 20));
                tc_fence_after();
#ifdef TNMF_TC_PROFILE
                const long long t_i = clock64();
#endif
                const unsigned ta = tmem_u + (unsigned)(p.a_col0 + st * kKS);
                if (elect_one()) {
#pragma unroll
                    for (int ks = 0; ks < kKS / 8; ++ks) {
                        const unsigned kb = (unsigned)ks * b_step16 + b0;
                        mma_tf32_ts2<true>(tset, ta + 8u * ks, b_lo_word | (ring_hi16 + kb), desc_hi, idesc);
                        mma_tf32_ts2<true>(tset, ta + 8u * ks, b_lo_word | (ring_lo16 + kb), desc_hi, idesc);
                    }
                }
                __syncwarp();
#ifdef TNMF_TC_PROFILE
                prof_issue += clock64() - t_i;
#endif
                mma_commit_elect(&a_empty[st]);
                if (++st == p.n_astages) { st = 0; ph ^= 1u; }
                // activation rows that leave the window: two per step, the whole window after the unit's last step
                for (int i = (q + 1 < w.steps) ? 2 : WP; i > 0; i -= 2) {
                    mma_commit_elect(&h_free[slot_out >> 1]);
                    slot_out += 2;
                    if (slot_out == RS) slot_out = 0;
                }
                slot_a += 2;
                if (slot_a >= RS) slot_a -= RS;
                if (++steps_done % kEpochSteps == 0) mma_commit_elect(&set_done[epoch & 1]);
            }
        }
        if (X < p.n_issue && steps_done % kEpochSteps != 0) mma_commit_elect(&set_done[(steps_done / kEpochSteps) & 1]);
#ifdef TNMF_TC_PROFILE
        prof_total += clock64();
        if (blockIdx.x == 0 && lane == 0 && X < p.n_issue)
            printf("gradw_ns mma %d: total %lld  wait a_full %lld  wait h_full %lld  wait set_free %lld  issuing %lld (%lld steps)\n", X, prof_total, prof_full, prof_hfull, prof_setfree, prof_issue, steps_done);
#endif
        __syncwarp();
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 8) tmem_dealloc(tmem_base, 512);
}

__global__ void __launch_bounds__(kThreads, 1) gradw_ns_kernel(const Geo2 g, const Plan p, const Args a) {
    gradw_ns_body<false>(g, p, a);
}
__global__ void __launch_bounds__(kThreads, 1) gradw_ns3_kernel(const Geo3 g, const Plan p, const Args a) {
    gradw_ns_body<true>(g, p, a);
}

}  // namespace gwn
}  // namespace tc

// ---- dispatch ----------------------------------------------------------------------------------------------------------
bool tc_gradw_ns_supported(const Geo &g, int dtype) {
    tc::gwn::Plan p;
    if (plane_problem(g)) return tc::plane_mode_ok(g, dtype) && tc::gwn::make_plan(tc::make_geo3(g, false), p);
    if (!tc::rank2_ok(g, dtype)) return false;
    return tc::gwn::make_plan(tiled::make_geo2(g), p);
}

size_t tc_gradw_ns_workspace_bytes(const Geo &g) {
    tc::gwn::Plan p;
    const bool planes = plane_problem(g);
    if (!(planes ? tc::gwn::make_plan(tc::make_geo3(g, false), p) : tc::gwn::make_plan(tiled::make_geo2(g), p))) return 0;
    return (size_t)p.grid * 4 * 2 * (size_t)g.M * g.C * (size_t)vol3(g.A) * sizeof(float);
}

int tc_gradient_w_ns(const Geo &g, const float *V, const float *R, const float *H, float *neg, float *pos, void *workspace,
                     size_t workspace_bytes, cudaStream_t st, int t_lo, int t_hi) {
    const bool planes = plane_problem(g);
    tc::Geo3 q3 = tc::make_geo3(g, false);
    const tiled::Geo2 q = planes ? q3 : tiled::make_geo2(g);
    tc::gwn::Plan p;
    if (!tc::gwn::make_plan(q, p)) return TNMF_EUNSUPPORTED;
    const long long count = (long long)g.M * g.C * vol3(g.A);
    if (!workspace || workspace_bytes < tc_gradw_ns_workspace_bytes(g)) return TNMF_EWORKSPACE;
    tc::gwn::Args a;
    a.V = V; a.R = R; a.H = H; a.partials = (float *)workspace;
    auto kern = tc::gwn::gradw_ns_kernel;
    auto kern3 = tc::gwn::gradw_ns3_kernel;
    cudaError_t e = cudaFuncSetAttribute(planes ? (const void *)kern3 : (const void *)kern,
                                         cudaFuncAttributeMaxDynamicSharedMemorySize, tc::gwn::kMaxSmem);
    if (e != cudaSuccess) return status_from_cuda(e);
    // A plane window [t_lo, t_hi): the pass of a_z covers the sample planes z whose activation plane z + offz - a_z lies
    // in it.  Its own plan has at most p.grid CTAs, and the CTAs (and a_z slices) it leaves out must read as zeros in the
    // fixed-order reduction over the p.grid * 4 slices: the partials are cleared first.  (The full window runs the
    // unwindowed launches.)
    const bool window = t_hi >= 0 && !(t_lo <= 0 && t_hi >= g.T[0]);
    if (window && !planes) return TNMF_EUNSUPPORTED;
    if (window) {
        cudaError_t e = cudaMemsetAsync(workspace, 0, tc_gradw_ns_workspace_bytes(g), st);
        if (e != cudaSuccess) return status_from_cuda(e);
    }
    // 3-D: one pass per atom plane a_z over the virtual samples (n, z), against H shifted by offz - a_z planes; each pass
    // fills its own a_z slice of every partial, and one fixed-order reduction finishes all of them
    for (int az = 0; az < (planes ? g.A[0] : 1); ++az) {
        q3.az = az;
        a.H = planes ? H + (long long)(q3.offz - az) * q3.hsz : H;
        tc::gwn::Plan pz = p;
        if (window) {
            const int z0 = max(0, t_lo - q3.offz + az), z1 = min(g.D[0], t_hi - q3.offz + az);
            if (z1 <= z0) continue;
            tc::window_geo3(q3, g.N, z0, z1 - z0);
            if (!tc::gwn::make_plan(q3, pz, p.grid)) return TNMF_EUNSUPPORTED;
        }
        for (int m0 = 0; m0 < g.M; m0 += tc::gwn::kNB) {
            a.m0 = m0;
            if (planes) kern3<<<(unsigned)pz.grid, tc::gwn::kThreads, pz.smem, st>>>(q3, pz, a);
            else kern<<<(unsigned)p.grid, tc::gwn::kThreads, p.smem, st>>>(q, p, a);
            TNMF_CHECK_LAUNCH();
        }
    }
    return finish_gradient_w<float>((const float *)workspace, p.grid * 4, count, neg, pos, st);
}

int tc_gradw_ns_launches(const Geo &g) { return g.A[0] * tiled::ceil_div(g.M, tc::gwn::kNB) + 1; }

}  // namespace tnmf
