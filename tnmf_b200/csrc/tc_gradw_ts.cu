// Tensor-core (tcgen05, 3xTF32) W gradient with the expanded operand in TENSOR MEMORY.
//
//   neg[m,c,ay,ax] = sum_n sum_{ty,tx} H[n,m,ty,tx] * Vext[n,c,ty-offy+ay,tx-offx+ax]      (tnmf/backends/NumPy.py:77-85)
//   pos[m,c,ay,ax] = the same with R                                                       (tnmf/backends/NumPy.py:80,87-90)
//
// Same product as tc_gradw.cu - a CTA owns 64 activation columns (column J = n * TXP + xv of the flattened [N x TXP] space,
// TXP = TX + AX - 1) and walks down the source rows r; per row
//       D'[k', (ay, m)] += sum_col A'[k', col] * B'[(ay, m), col],   k' = (X, c, ax), X in {V, R}
//       A'[(X, c, ax), col] = Xext[n, c, r, xv - offx + ax]          B'[(slot, m), col] = H[n, m, ty(slot), xv]
// with the activation rows B' in a shared-memory ring and the accumulator (lane = k', column = (ay, m)) resident in TMEM -
// but A' never exists in shared memory: it is an operand in TENSOR MEMORY, lane = k', column = tile column.  The thread that
// owns lane (X, c, ax) reads its shifted copy of the raw source row (conflict-free LDS.32: consecutive lanes, consecutive
// words), splits hi/lo in registers and writes 16 columns with one tcgen05.st per half.  What that buys (measured,
// tools/tc_probe2.cu and profiles/r02_*): the MMA no longer fetches a 4 KB A operand over the shared-memory port per
// instruction (it was 45 % of the port's traffic), the expansion's STS.128 and its 70 % bank-conflict rate are gone, and the
// operand lanes need no padding to 8-row core matrices.
//
// TMEM columns: two accumulator sets of NA = 16 * AY columns (a chain is cut after kEpoch source rows because the tensor
// core truncates when it adds into the accumulator; while one set accumulates, the other is added into the CTA's slice in
// global memory and zeroed), then the operand stages: KS columns of hi + KS of lo each (KS = 32 or 16 tile columns).
// V taps sit in lanes [0, C*AX), R taps in lanes [64, 64 + C*AX), so all four lane quarters have writers.
//
// Roles (448 threads): warps 0-7 workers (warp w writes lane quarter w % 4, column half w / 4 of a stage; together they stage
// the raw rows and the new activation row), warps 8 and 9 issue the MMAs, each for a FIXED half of the atom rows
// (converged warps, one elected lane; the live-row window is always one run of ring slots: the first AY - 1 slots are stored
// a second time behind the last one), warps 10-13 drain the sets.  A TMEM column is written by one warp only, so the order
// of accumulation is fixed: two warps whose split followed the ring's wrap-around made a column change hands between source
// rows and their relative progress decide which row was added first - run-to-run differences of one ulp (found by
// tools/determinism_check.py; the tensor core truncates, so the order matters).  The same happens when two warps take
// strict turns on the same columns: MMAs of different warps are not executed in the order they were issued.  mbarriers: a_full/a_empty per operand stage,
// h_full/h_free per ring slot, set_done/set_free per accumulator set.  Atoms in blocks of 16 (one launch per block).
#include "tc_common.cuh"

namespace tnmf {
namespace tc {
namespace gwt {

using tiled::ceil_div;
using tiled::Geo2;
using tiled::round_up;

constexpr int kCT = 64;             // activation columns per tile
constexpr int kNB = 16;             // atoms per launch
constexpr int kWorkers = 256;
#ifndef TNMF_GW_ISSUERS
#define TNMF_GW_ISSUERS 2
#endif
constexpr int kIssuers = TNMF_GW_ISSUERS;   // issuing warps, each owning a FIXED share of the atom rows (= accumulator columns)
constexpr int kThreads = 32 * (8 + kIssuers + 4);
constexpr int kEpoch = 8;           // source rows accumulated into one TMEM set before it is drained
constexpr int kMaxAStages = 4;
constexpr int kRingMax = 24;
constexpr int kRawMax = 4;          // raw elements per worker: 2 * C * (64 + AX - 1) <= 1024
constexpr int kMaxSmem = 226 * 1024;

struct Plan {
    int KPL;                        // taps per plane = C * AX (<= 64)
    int TXP, RW, RWp, rawX, raw_floats, nraw;
    int KS, n_sub, n_astages, a_col0, NA;
    int RS, NRr, ring_floats;       // logical ring slots, physical ring rows (16 per slot, RS + AY - 1 slots: the first
                                    // AY - 1 slots are mirrored behind the last one), floats of ONE of the hi / lo halves
    int tiles;
    long long total, quota, units;  // tile-rows of the problem, tile-rows per CTA, grid * (most segments of a CTA)
    int round_robin;                // 1: unit u is the whole tile u (CTA u % grid); 0: linear ranges
    int grid;
    size_t smem;
};

struct Args {
    const float *V, *R, *H;
    float *partials;                // [grid][2][M*C*AY*AX]
    int m0;
};

bool make_plan(const Geo2 &g, Plan &p) {
    p = Plan();
    if (g.AY < 1 || g.AY > 14) return false;
    p.KPL = g.C * g.AX;
    if (p.KPL > 64) return false;
    p.NA = kNB * g.AY;
    const int spare = 512 - 2 * p.NA;
#ifdef TNMF_GW_KS16
    if (spare >= 2 * 32) p.KS = 16;
#else
    if (spare >= 2 * 64) p.KS = 32;
#endif
    else if (spare >= 2 * 32) p.KS = 16;
    else return false;
    p.n_sub = kCT / p.KS;
    p.n_astages = spare / (2 * p.KS);
    if (p.n_astages > kMaxAStages) p.n_astages = kMaxAStages;
    p.n_astages &= ~1;                                      // even: an operand stage always belongs to the same issuing warp
    p.a_col0 = 2 * p.NA;
    p.TXP = g.TX + g.AX - 1;
    p.RW = kCT + g.AX - 1;
    // channel pitch == AX (mod 32): lane k = (c, ax) then reads word c * RWp + ax + col == k + col (mod 32): no bank conflicts
    p.RWp = p.RW + 1;
    while ((p.RWp - g.AX) % 32 != 0) ++p.RWp;
    p.rawX = round_up(g.C * p.RWp, 32);
    p.raw_floats = 2 * p.rawX + 128;                        // V plane, R plane, zeros for the idle lanes
    p.nraw = ceil_div(2 * g.C * p.RW, kWorkers);
    if (p.nraw > kRawMax) return false;
    const size_t fixed = (size_t)2 * p.raw_floats * 4 + 1024;
    for (p.RS = kRingMax; p.RS >= g.AY + 1; --p.RS) {
        p.NRr = (p.RS + g.AY - 1) * kNB;
        p.ring_floats = (p.NRr * 4 + 4) * (kCT / 4);        // K-chunk stride padded by 16 bytes: conflict-free row staging
        if (fixed + (size_t)2 * p.ring_floats * 4 <= (size_t)kMaxSmem) break;
    }
    if (p.RS < g.AY + 1) return false;
    p.smem = fixed + (size_t)2 * p.ring_floats * 4;
    const long long cols = (long long)g.N * p.TXP;
    if (cols <= 0 || cols >= (1ll << 31) - kCT) return false;
    p.tiles = (int)((cols + kCT - 1) / kCT);
    // Work split: the (tile, row) space is cut into `grid` equal LINEAR ranges, one per CTA (a range is a few row segments
    // of consecutive tiles) - every SM gets the same number of rows whatever the number of tiles (cfg2: 138 / 145 / 276
    // tiles on 148 SMs left 7 - 10 % of the SMs idle with whole-tile units).  A segment boundary costs AY - 1 extra source
    // rows, and there are at most two per CTA.
    const int sms = tma::sm_count();
    p.total = (long long)p.tiles * g.TY;
    p.quota = (p.total + sms - 1) / sms;
    const long long min_quota = g.TY < 8 ? g.TY : 8;
    if (p.quota < min_quota) p.quota = min_quota;
    // Whole tiles, dealt ROUND-ROBIN, when that costs little: the CTAs then work on consecutive tiles and walk down the same
    // rows at the same time, so the tiles of a sample share its V / R rows (and the activation sectors at tile borders) in
    // L2.  ncu, cfg2: 394 MB of DRAM reads per launch this way against 580 - 600 MB when every CTA owns a contiguous range
    // of the (tile, row) space, for 1.4 % of kernel time.
    const long long whole = (p.tiles + sms - 1) / sms * (long long)g.TY;
    p.round_robin = (double)whole <= 1.1 * (double)(p.quota + 2 * (g.AY - 1));
    if (p.round_robin) {
        p.quota = g.TY;
        p.grid = p.tiles < sms ? p.tiles : sms;
        p.units = p.tiles;
        return true;
    }
    p.grid = (int)((p.total + p.quota - 1) / p.quota);
    p.units = (long long)p.grid * ((p.quota + g.TY - 2) / g.TY + 1);
    return true;
}

struct Unit {
    int tile, ty0, ty1, r_lo, r_hi;
};
__device__ __forceinline__ Unit make_unit(long long u, const Geo2 &g, const Plan &p) {
    // unit u = segment u / grid of CTA u % grid (gridDim.x == p.grid); empty (ty0 == ty1) past the CTA's last segment
    Unit w;
    const long long b = u % p.grid, k = u / p.grid;
    const long long lo = p.round_robin ? u * (long long)g.TY : b * p.quota, hi = min(lo + p.quota, p.total);
    w.tile = p.round_robin ? (int)u : (int)(lo / g.TY + k);
    const long long t0 = (long long)w.tile * g.TY;
    const long long s0 = max(lo, t0), s1 = min(hi, t0 + g.TY);
    w.ty0 = s1 > s0 ? (int)(s0 - t0) : 0;
    w.ty1 = s1 > s0 ? (int)(s1 - t0) : 0;
    w.r_lo = max(0, w.ty0 - g.offy);
    w.r_hi = min(g.DY - 1, w.ty1 - 1 - g.offy + g.AY - 1);
    return w;
}

// KS: tile columns per operand stage (32: every worker thread writes 16 columns per half, 16: 8 columns)
template <int KS>
__global__ void __launch_bounds__(kThreads, 1) gradw_ts_kernel(const Geo2 g, const Plan p, const Args a) {
    extern __shared__ __align__(128) float smem[];
    __shared__ __align__(8) unsigned long long a_full[kMaxAStages], a_empty[kMaxAStages], h_full[kRingMax], h_free[kRingMax],
        set_done[2], set_free[2];
    __shared__ unsigned tmem_base_s;
    constexpr int CPT = KS / 2;                                  // columns per worker thread and stage
    // the warp index comes out of a shuffle so that ptxas knows it is warp-uniform: the role branches below then are
    // uniform branches and the code inside them may live in uniform registers (what the tcgen05 operands need)
    const int tid = threadIdx.x, warp = __shfl_sync(0xffffffffu, tid >> 5, 0), lane = tid & 31;
    const int AY = g.AY, AX = g.AX, C = g.C, RS = p.RS, RW = p.RW;
    float *ring_hi = smem, *ring_lo = smem + p.ring_floats;
    float *raw = ring_lo + p.ring_floats;                       // [2 buffers][V plane | R plane | zeros]

    if (tid == 0) {
        for (int s = 0; s < p.n_astages; ++s) { mbar_init(&a_full[s], 8); mbar_init(&a_empty[s], kIssuers); }
        for (int s = 0; s < kRingMax; ++s) { mbar_init(&h_full[s], kWorkers); mbar_init(&h_free[s], kIssuers); }
        for (int s = 0; s < 2; ++s) { mbar_init(&set_done[s], kIssuers); mbar_init(&set_free[s], 128); }
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

    const long long count = (long long)g.M * C * AY * AX;

    if (warp < 8) {
        // ------------------------------------ workers ------------------------------------
        const int quarter = warp & 3, half = warp >> 2;
        const int L = quarter * 32 + lane;                      // operand lane of this thread
        const int X = L >> 6, k = L & 63;
        const bool live = k < p.KPL;
        const bool warp_live = ((quarter * 32) & 63) < p.KPL;   // lane 0 of the warp carries a tap
        const int src_off = live ? X * p.rawX + (k / AX) * p.RWp + (k % AX) : 2 * p.rawX + 16;   // idle lanes: zeros, in the
                                                                                              // bank a live lane 32 does not use
        const unsigned t_lane = tmem_base + ((unsigned)(quarter * 32) << 16) + (unsigned)(p.a_col0 + half * CPT);
        int st = 0;
        unsigned ph = 0, buf = 0;
        TC_PROF_DECL(empty); TC_PROF_DECL(hfree); TC_PROF_DECL(bar); TC_PROF_DECL(total);
#ifdef TNMF_TC_PROFILE
        prof_total = -clock64();
#endif
        const long long plane = (long long)g.DY * g.DX;
        const int raw_count = 2 * C * RW;
        const int h_ml = tid >> 4, h_cg = tid & 15;             // activation chunk: atom ml, columns 4 cg .. 4 cg + 3
        int slot_new = 0;                                       // ring slot of the next activation row; no divisions in
        unsigned wraps = 0;                                     // the row loop (they were most of its critical path)
        for (long long u = blockIdx.x; u < p.units; u += gridDim.x) {
            const Unit w = make_unit(u, g, p);
            if (w.ty0 >= w.ty1) break;                            // past this CTA's last segment
            // source element of every raw slot (q = tid + 256 e -> tensor, channel, position) in row 0, or -1: zero
            long long roff[kRawMax];
            int rdst[kRawMax];
#pragma unroll
            for (int e = 0; e < kRawMax; ++e) {
                roff[e] = -1;
                rdst[e] = -1;
                const int q = tid + kWorkers * e;
                if (e < p.nraw && q < raw_count) {
                    const int Xq = q / (C * RW), qq = q - Xq * (C * RW);
                    const int c = qq / RW, xr = qq - c * RW;
                    rdst[e] = Xq * p.rawX + c * p.RWp + xr;
                    const long long J = (long long)w.tile * kCT + xr;
                    const int n = (int)(J / p.TXP);
                    const int x = (int)(J - (long long)n * p.TXP) - g.offx;
                    if (n < g.N && (unsigned)x < (unsigned)g.DX) roff[e] = ((long long)n * C + c) * plane + x;
                }
            }
            long long hoff[4];
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const long long J = (long long)w.tile * kCT + 4 * h_cg + e;
                const int n = (int)(J / p.TXP);
                const int xv = (int)(J - (long long)n * p.TXP);
                hoff[e] = (n < g.N && xv < g.TX && a.m0 + h_ml < g.M)
                              ? (long long)n * g.hsn + (long long)(a.m0 + h_ml) * g.hsm + xv : -1;
            }
            float rv[kRawMax];
            auto load_raw = [&](int r) {
#pragma unroll
                for (int e = 0; e < kRawMax; ++e) {
                    const float *src = ((tid + kWorkers * e) >= C * RW) ? a.R : a.V;
                    rv[e] = roff[e] >= 0 ? __ldg(src + (long long)r * g.DX + roff[e]) : 0.f;
                }
            };
            auto load_h = [&](int ty) {
                float4 hv;
                hv.x = hoff[0] >= 0 ? a.H[hoff[0] + (long long)ty * g.hsy] : 0.f;
                hv.y = hoff[1] >= 0 ? a.H[hoff[1] + (long long)ty * g.hsy] : 0.f;
                hv.z = hoff[2] >= 0 ? a.H[hoff[2] + (long long)ty * g.hsy] : 0.f;
                hv.w = hoff[3] >= 0 ? a.H[hoff[3] + (long long)ty * g.hsy] : 0.f;
                return hv;
            };
            float4 hv_next = make_float4(0.f, 0.f, 0.f, 0.f);
            int hv_row = -1;
            int next_new = w.ty0;
            load_raw(w.r_lo);
            for (int r = w.r_lo; r <= w.r_hi; ++r) {
                // ---- activation rows that enter the window with this source row ----
                const int t_b = min(w.ty1 - 1, r + g.offy);
                unsigned new_slots = 0;
                for (; next_new <= t_b; ++next_new) {
                    const int slot = slot_new;
                    const float4 hv = next_new == hv_row ? hv_next : load_h(next_new);
                    if (wraps) TC_PROF_WAIT(hfree, mbar_wait_backoff(&h_free[slot], (wraps - 1u) & 1u, 40));
                    if (++slot_new == RS) { slot_new = 0; ++wraps; }
                    float4 hi, lo;
                    split_tf32(hv.x, hi.x, lo.x); split_tf32(hv.y, hi.y, lo.y);
                    split_tf32(hv.z, hi.z, lo.z); split_tf32(hv.w, hi.w, lo.w);
                    const int nrow = slot * kNB + h_ml;
                    const size_t o = (size_t)(nrow >> 3) * 32 + (size_t)h_cg * (p.NRr * 4 + 4) + (size_t)(nrow & 7) * 4;
                    *reinterpret_cast<float4 *>(ring_hi + o) = hi;
                    *reinterpret_cast<float4 *>(ring_lo + o) = lo;
                    if (slot < AY - 1) {                                // mirror: a window never wraps (one MMA per K step)
                        const size_t om = o + (size_t)RS * (kNB / 8) * 32;
                        *reinterpret_cast<float4 *>(ring_hi + om) = hi;
                        *reinterpret_cast<float4 *>(ring_lo + om) = lo;
                    }
                    new_slots |= 1u << slot;
                }
                if (new_slots) {
                    fence_proxy_async();
                    for (; new_slots; new_slots &= new_slots - 1) mbar_arrive(&h_full[__ffs(new_slots) - 1]);
                }
                // ---- raw V and R rows of this tile (plain FP32; split when they are expanded) ----
                float *rb = raw + (size_t)buf * p.raw_floats;
#pragma unroll
                for (int e = 0; e < kRawMax; ++e)
                    if (rdst[e] >= 0) rb[rdst[e]] = rv[e];
                if (r < w.r_hi) load_raw(r + 1);                    // in flight while this row is expanded
                if (next_new < w.ty1) { hv_next = load_h(next_new); hv_row = next_new; }
                TC_PROF_WAIT(bar, asm volatile("bar.sync 1, 256;\n" ::: "memory"));
                // ---- expansion into tensor memory: lane (X, c, ax) <- raw[X][c][ax + col] ----
                const float *src = rb + src_off + half * CPT;
                for (int h = 0; h < kCT / KS; ++h) {
                    TC_PROF_WAIT(empty, mbar_wait_backoff(&a_empty[st], ph ^ 1u, 20));
                    tc_fence_after();
                    if (warp_live) {
                        float hi[CPT], lo[CPT];
#pragma unroll
                        for (int j = 0; j < CPT; ++j) split_tf32(src[h * KS + j], hi[j], lo[j]);
                        const unsigned t = t_lane + (unsigned)(st * 2 * KS);
                        if constexpr (CPT == 16) {
                            tmem_st16(t, hi);
                            tmem_st16(t + KS, lo);
                        } else {
                            tmem_st8(t, hi);
                            tmem_st8(t + KS, lo);
                        }
                        tmem_st_wait();
                    }
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(&a_full[st]);
                    if (++st == p.n_astages) { st = 0; ph ^= 1u; }
                }
                buf ^= 1u;
            }
        }
#ifdef TNMF_TC_PROFILE
        prof_total += clock64();
        if (blockIdx.x == 0 && tid == 0)
            printf("gradw_ts workers: total %lld  wait a_empty %lld  wait h_free %lld  raw barrier %lld\n", prof_total, prof_empty,
                   prof_hfree, prof_bar);
#endif
    } else if (warp >= 8 + kIssuers) {
        // ------------------------------------ accumulator drainers ------------------------------------
        int rows_done = 0;
        bool first_drain = true;
        TC_PROF_DECL(done); TC_PROF_DECL(total);
#ifdef TNMF_TC_PROFILE
        prof_total = -clock64();
#endif
        auto drain = [&](int e) {
            const int set = (int)(e & 1);
            const int l = (warp & 3) * 32 + lane;
            const int X = l >> 6, k = l & 63;
            const bool live = k < p.KPL;
            const int c = live ? k / AX : 0, ax = live ? k - c * AX : 0;
            float *slice = a.partials + (long long)blockIdx.x * 2 * count + (long long)X * count;
            const unsigned tbase = tmem_base + ((unsigned)((warp & 3) * 32) << 16) + (unsigned)(set * p.NA);
            float old_next[kNB];
#pragma unroll
            for (int ml = 0; ml < kNB; ++ml) old_next[ml] = 0.f;
            if (live && !first_drain) {
                const float *nx = slice + (((long long)a.m0 * C + c) * AY + (AY - 1)) * AX + ax;
#pragma unroll
                for (int ml = 0; ml < kNB; ++ml) old_next[ml] = a.m0 + ml < g.M ? __ldcg(nx + ml * (long long)C * AY * AX) : 0.f;
            }
            TC_PROF_WAIT(done, mbar_wait_backoff(&set_done[set], (unsigned)((e >> 1) & 1), 100));
            tc_fence_after();
            // The running sums of the slice do not depend on the set: those of window position 0 were fetched before the
            // wait above, those of position j + 1 are fetched while position j is added (a drain used to cost 11 dependent
            // round trips to L2, 22 k clk per epoch against 17 k clk of MMAs: the drainers set the pace).
            const long long mstride = (long long)C * AY * AX;
            float *dst_base = slice + (((long long)a.m0 * C + c) * AY) * AX + ax;
            for (int j = 0; j < AY; ++j) {
                float v[16], old[kNB];
#pragma unroll
                for (int ml = 0; ml < kNB; ++ml) old[ml] = old_next[ml];
                if (j + 1 < AY && live && !first_drain) {
                    const float *nx = dst_base + (long long)(AY - 2 - j) * AX;
#pragma unroll
                    for (int ml = 0; ml < kNB; ++ml) old_next[ml] = a.m0 + ml < g.M ? __ldcg(nx + ml * mstride) : 0.f;
                }
                tmem_ld16(tbase + (unsigned)(j * kNB), v);
                tmem_ld_wait();
                tmem_st16_zero(tbase + (unsigned)(j * kNB));
                if (live) {
                    float *dst0 = dst_base + (long long)(AY - 1 - j) * AX;
#pragma unroll
                    for (int ml = 0; ml < kNB; ++ml)
                        if (a.m0 + ml < g.M) __stcg(dst0 + ml * mstride, v[ml] + old[ml]);
                }
            }
            tmem_st_wait();
            tc_fence_before();
            mbar_arrive(&set_free[set]);
            first_drain = false;
        };
        for (long long u = blockIdx.x; u < p.units; u += gridDim.x) {
            const Unit w = make_unit(u, g, p);
            if (w.ty0 >= w.ty1) break;                            // past this CTA's last segment
            rows_done += w.r_hi - w.r_lo + 1;
        }
        const int n_epochs = (rows_done + kEpoch - 1) / kEpoch;
        for (int e = 0; e < n_epochs; ++e) drain(e);
#ifdef TNMF_TC_PROFILE
        prof_total += clock64();
        if (blockIdx.x == 0 && tid == 32 * (8 + kIssuers))
            printf("gradw_ts drainers: total %lld  wait set_done %lld  (%d epochs)\n", prof_total, prof_done, n_epochs);
#endif
    } else {
        // ------------------------------------ MMA issuer (one converged warp, one elected lane) ------------------------------------
        // everything an MMA names must sit in UNIFORM registers: a value ptxas cannot prove warp-uniform costs an R2UR per
        // operand and instruction (35 instructions per MMA, measured: the issuing warp, not the tensor pipe, set the pace).
        // A shuffle from lane 0 is the idiom that marks a loaded value as uniform.
        const unsigned tmem_u = __shfl_sync(0xffffffffu, tmem_base, 0);
        const unsigned lbo_b = (unsigned)p.NRr * 16 + 16;       // ring chunks carry a 16-byte pad
        const unsigned desc_hi = (128u >> 4) | (1u << 14);      // SBO, descriptor version 1
        const unsigned b_lo_word = ((lbo_b >> 4) << 16);
        const unsigned ring_hi16 = __shfl_sync(0xffffffffu, smem_u32(ring_hi) >> 4, 0);
        const unsigned ring_lo16 = __shfl_sync(0xffffffffu, smem_u32(ring_lo) >> 4, 0);
        const unsigned b_step16 = (2 * lbo_b) >> 4;
        // Warp X owns the window positions (= atom rows = accumulator column blocks) [j_lo, j_hi]: a TMEM column is only ever
        // written by one warp, in program order - bitwise reproducible however the two warps interleave - and what one warp
        // spends between two rows (barrier waits, commits, bookkeeping: ~1000 clk, during which the two-or-three-deep MMA
        // queue of a single issuer ran dry) is hidden behind the other warp's MMAs.  The split is static because the
        // mirrored ring never splits a window; a split that moved with the ring's wrap-around made columns change hands
        // between rows and the accumulation order timing dependent (one-ulp run-to-run differences).
        const int X = warp - 8;
        const int j_lo = (AY * X + kIssuers - 1) / kIssuers, j_hi = (AY * (X + 1) + kIssuers - 1) / kIssuers - 1;
        int st = 0;
        unsigned ph = 0;
        int rows_done = 0;
        // ring bookkeeping without divisions: slot / wrap parity of the next row to enter, slot of the next row to leave,
        // slot of the first row of the window
        int slot_new = 0, slot_out = 0, slot_a = 0;
        unsigned par_new = 0;
        TC_PROF_DECL(full); TC_PROF_DECL(hfull); TC_PROF_DECL(setfree); TC_PROF_DECL(total); TC_PROF_DECL(issue); TC_PROF_DECL(commit); TC_PROF_DECL(commit2);
#ifdef TNMF_TC_PROFILE
        prof_total = -clock64();
#endif
        for (long long u = blockIdx.x; u < p.units; u += gridDim.x) {
            const Unit w = make_unit(u, g, p);
            if (w.ty0 >= w.ty1) break;                            // past this CTA's last segment
            int next_new = w.ty0, next_out = w.ty0, win0 = w.ty0;
            slot_a = slot_new;                                      // the unit's first activation row enters here
            for (int r = w.r_lo; r <= w.r_hi; ++r) {
                const int epoch = rows_done / kEpoch;
                if (rows_done % kEpoch == 0 && epoch >= 2) {
                    TC_PROF_WAIT(setfree, mbar_wait(&set_free[epoch & 1], (unsigned)(((epoch >> 1) - 1) & 1)));
                    tc_fence_after();
                }
                const unsigned tset = tmem_u + (unsigned)((epoch & 1) * p.NA);
                const int ay_hi = min(AY - 1, r + g.offy - w.ty0);
                const int t_a = r + g.offy - ay_hi, t_b = min(w.ty1 - 1, r + g.offy);
                const int j0 = r + g.offy - AY + 1;                 // activation row of accumulator column block 0
                for (; next_new <= t_b; ++next_new) {
                    TC_PROF_WAIT(hfull, mbar_wait(&h_full[slot_new], par_new));
                    if (++slot_new == RS) { slot_new = 0; par_new ^= 1u; }
                }
                for (; win0 < t_a; ++win0)
                    if (++slot_a == RS) slot_a = 0;
                // the window [t_a, t_b] is ONE run of physical ring slots (the head of the ring is mirrored behind its tail);
                // this warp's part of it: [ta_x, tb_x]
                const int ta_x = max(t_a, j0 + j_lo), tb_x = min(t_b, j0 + j_hi);
                const int cnt = tb_x - ta_x + 1;
                const unsigned col0 = tset + (unsigned)((ta_x - j0) * kNB);
                const unsigned idesc0 = idesc_tf32(128, kNB * max(cnt, 1));
                const unsigned b0 = (unsigned)(slot_a + (ta_x - t_a)) * 16u;
                for (int h = 0; h < kCT / KS; ++h) {
                    TC_PROF_WAIT(full, mbar_wait(&a_full[st], ph));
                    tc_fence_after();
#ifdef TNMF_TC_PROFILE
                    const long long t_i = clock64();
#endif
                    const unsigned ta_hi = tmem_u + (unsigned)(p.a_col0 + st * 2 * KS), ta_lo = ta_hi + KS;
                    if (cnt > 0 && elect_one()) {
#pragma unroll
                        for (int ks = 0; ks < KS / 8; ++ks) {
                            const unsigned kb = (unsigned)(h * (KS / 8) + ks) * b_step16 + b0;
                            const unsigned long long b_hi = ((unsigned long long)desc_hi << 32) | (b_lo_word | (ring_hi16 + kb));
                            const unsigned long long b_lo = ((unsigned long long)desc_hi << 32) | (b_lo_word | (ring_lo16 + kb));
                            mma_tf32_ts(col0, ta_hi + 8u * ks, b_hi, idesc0, 1u);
                            mma_tf32_ts(col0, ta_lo + 8u * ks, b_hi, idesc0, 1u);
                            mma_tf32_ts(col0, ta_hi + 8u * ks, b_lo, idesc0, 1u);
                        }
                    }
                    __syncwarp();
#ifdef TNMF_TC_PROFILE
                    prof_issue += clock64() - t_i;
#endif
                    TC_PROF_WAIT(commit, mma_commit_elect(&a_empty[st]));
                    if (++st == p.n_astages) { st = 0; ph ^= 1u; }
                }
                // activation rows that leave the window: their slots may be overwritten once these MMAs are done (both
                // warps commit: h_free counts two arrivals, each commit covers the committing warp's own MMAs)
                for (; next_out < w.ty1 && min(g.DY - 1, next_out - g.offy + AY - 1) <= r; ++next_out) {
                    TC_PROF_WAIT(commit2, mma_commit_elect(&h_free[slot_out]));
                    if (++slot_out == RS) slot_out = 0;
                }
                if (++rows_done % kEpoch == 0) mma_commit_elect(&set_done[epoch & 1]);
            }
        }
        if (rows_done % kEpoch != 0) mma_commit_elect(&set_done[(rows_done / kEpoch) & 1]);
#ifdef TNMF_TC_PROFILE
        prof_total += clock64();
        if (blockIdx.x == 0 && lane == 0)
            printf("gradw_ts mma %d: total %lld  wait a_full %lld  wait h_full %lld  wait set_free %lld  issuing %lld  commit a_empty %lld  commit h_free %lld (%d rows)\n",
                   X, prof_total, prof_full, prof_hfull, prof_setfree, prof_issue, prof_commit, prof_commit2, rows_done);
#endif
        __syncwarp();
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 8) tmem_dealloc(tmem_base, 512);
}

template <int KS>
static int launch(const Geo2 &g, const Plan &p, const Args &a, cudaStream_t st) {
    auto kern = gradw_ts_kernel<KS>;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, kMaxSmem);
    if (e != cudaSuccess) return status_from_cuda(e);
    kern<<<(unsigned)p.grid, kThreads, p.smem, st>>>(g, p, a);
    TNMF_CHECK_LAUNCH();
    return TNMF_OK;
}

}  // namespace gwt
}  // namespace tc

// ---- dispatch ----------------------------------------------------------------------------------------------------------
bool tc_gradw_ts_supported(const Geo &g, int dtype) {
    if (!tc::rank2_ok(g, dtype)) return false;
    tc::gwt::Plan p;
    return tc::gwt::make_plan(tiled::make_geo2(g), p);
}

size_t tc_gradw_ts_workspace_bytes(const Geo &g) {
    tc::gwt::Plan p;
    if (!tc::gwt::make_plan(tiled::make_geo2(g), p)) return 0;
    return (size_t)p.grid * 2 * (size_t)g.M * g.C * g.A[1] * g.A[2] * sizeof(float);
}

int tc_gradient_w_ts(const Geo &g, const float *V, const float *R, const float *H, float *neg, float *pos, void *workspace,
                     size_t workspace_bytes, cudaStream_t st) {
    const tiled::Geo2 q = tiled::make_geo2(g);
    tc::gwt::Plan p;
    if (!tc::gwt::make_plan(q, p)) return TNMF_EUNSUPPORTED;
    const long long count = (long long)g.M * g.C * g.A[1] * g.A[2];
    if (!workspace || workspace_bytes < tc_gradw_ts_workspace_bytes(g)) return TNMF_EWORKSPACE;
    tc::gwt::Args a;
    a.V = V; a.R = R; a.H = H; a.partials = (float *)workspace;
    for (int m0 = 0; m0 < g.M; m0 += tc::gwt::kNB) {
        a.m0 = m0;
        const int s = p.KS == 32 ? tc::gwt::launch<32>(q, p, a, st) : tc::gwt::launch<16>(q, p, a, st);
        if (s) return s;
    }
    return finish_gradient_w<float>((const float *)workspace, p.grid, count, neg, pos, st);
}

int tc_gradw_ts_launches(const Geo &g) { return tiled::ceil_div(g.M, tc::gwt::kNB) + 1; }

}  // namespace tnmf
