// Tensor-core (tcgen05, 3xTF32) W gradient: a split-K reduction over samples and positions.
//
//   neg[m,c,ay,ax] = sum_n sum_{ty,tx} H[n,m,ty,tx] * Vext[n,c,ty-offy+ay,tx-offx+ax]      (tnmf/backends/NumPy.py:77-85)
//   pos[m,c,ay,ax] = the same with R                                                       (tnmf/backends/NumPy.py:80,87-90)
//
// Formulation (the transposed product of tc_hupd.cu).  A CTA owns a tile of 64 activation COLUMNS - column J = n * TXP + xv
// of the flattened [N x TXP] space, TXP = TX + AX - 1 (gap columns carry zero activations) - and walks down the rows.
// For a source row r the workers build, once, the expanded rows of V and of R stacked into ONE operand
//       A'[k', col]   k' = (X, c, ax), X in {V, R}:  A'[.., col] = Xext[n, c, r, xv - offx + ax]         2*KP x 64, K-major
// and keep the activation rows that meet r, ty = r + offy - ay, in a ring of AY + 1 row tiles
//       B'[(slot, m), col] = H[n, m, ty(slot), xv]                                                      16 rows per slot
// One tcgen05.mma (M = 128 lanes of which 2*KP carry taps, N = 16 atoms x live rows, K = 8 columns) then accumulates
//       D'[k', (ay, m)] += sum_col A'[k', col] * B'[(ay, m), col]
// for all atom rows of the source row at once; the accumulator (128 lanes x 16*AY columns) stays in TMEM for the whole
// life of the CTA - numerator in lanes [0, KP), denominator in lanes [KP, 2 KP) - and is written out once as one
// partial slice per CTA; finish_gradient_w sums the slices in a fixed order in double (deterministic, no atomics).
// 3xTF32: hi*hi + lo*hi + hi*lo, FP32 accumulation in TMEM.  The tensor core TRUNCATES when it adds into the
// accumulator (measured: 3e-8 relative bias per accumulation), so a chain is cut after kEpoch source rows: two
// accumulator sets alternate in TMEM and while one accumulates, the finished one is added (FP32 round-to-nearest) into
// the CTA's slice in global memory and zeroed.  The MMA reads 128 operand rows; rows past 2*KP alias the
// following K chunk (finite values, their accumulator lanes are never read).
//
// Roles (448 threads): warps 0-7 workers (stage the new activation row into the ring, expand V and R), warps 8 and 9
// issue the MMAs of the two runs of the live-row window (converged warps, one elected lane each), warps 10-13 drain the sets.  mbarriers: a_full/a_empty per operand stage, h_full/h_free per ring slot, set_done/set_free per set.
// Atoms in blocks of 16 (one launch per block).  Bound: tensor pipe at the TF32 rate / 3 with 2*KP/128 useful lanes.
#include <cstdlib>
#include "tc_common.cuh"

namespace tnmf {
namespace tc {

using tiled::ceil_div;
using tiled::Geo2;
using tiled::round_up;

namespace gw {

#ifndef TNMF_GW_EPOCH
#define TNMF_GW_EPOCH 8
#endif
// ONE issuing warp: with two, the window was cut where the ring wraps, so an accumulator column changed hands between
// source rows and the tensor pipe does not execute the MMAs of different warps in issue order - the truncating
// accumulation then depended on timing (tools/determinism_check.py: one-ulp run-to-run differences; tc_gradw_ts.cu avoids
// it with a mirrored ring and a static split).  This kernel is the fallback form now: it pays ~7 % for being bitwise
// reproducible.
#ifndef TNMF_GW_ISSUERS
#define TNMF_GW_ISSUERS 1
#endif
constexpr int kCT = 64;             // activation columns per tile = contraction length of one source row
constexpr int kNB = 16;             // atoms per launch
constexpr int kWorkers = 256;
constexpr int kThreads = 32 * (8 + TNMF_GW_ISSUERS + 4);   // 8 workers + MMA issuers + 4 accumulator drainers
constexpr int kEpoch = TNMF_GW_EPOCH;  // source rows accumulated into one TMEM set before it is drained
constexpr int kIssuers = TNMF_GW_ISSUERS;
constexpr int kMaxStages = 4;
constexpr int kMaxSmem = 226 * 1024;
constexpr int kRawMax = 4;          // raw elements per worker and tensor pair: 2 * C * (64 + AX - 1) <= 1024
constexpr int kRingMax = 18;        // ring slots (activation rows resident in shared memory)
constexpr int kChunkMax = 8;        // 16-byte chunks of an operand stage per worker: 2 * KP * 16 <= 2048

struct Plan {
    int KP, TXP, RW, raw_floats, nraw, nchunk;
    int S, NP;                      // source rows stacked into one operand, operand planes = 2 S (row, V | R)
    int RS, NRr;                    // ring slots (AY + 1), ring rows (16 per slot)
    int ring_floats, stage_floats;  // floats of ONE of the hi / lo halves
    int tiles, rblocks, rows_per_block;
    long long units;
    int n_stages, grid;
    size_t smem;
};

struct Args {
    const float *V, *R, *H;
    float *partials;                // [grid][S][2][M*C*AYW*AX]
    int m0;
    int ay0, AYW;                   // atom rows [ay0, ay0 + g.AY) of an atom AYW rows high (tall atoms run in row chunks)
    int accumulate;                 // 1: the slices were zeroed by the host and every drain adds (several launches share them)
};

bool make_plan(const Geo2 &g, Plan &p) {
    p = Plan();
    if (g.AY < 1 || g.AY > 15) return false;
    p.KP = round_up(g.C * g.AX, 8);
    if (2 * p.KP > 128) return false;
    p.TXP = g.TX + g.AX - 1;
    p.RW = kCT + g.AX - 1;
    p.raw_floats = round_up(g.C * p.RW + kCT + 8, 32);      // + zeros read by the padded k
    // narrow atoms (C*AX <= 32) leave most of the 128 MMA lanes empty: stack two consecutive source rows, whose
    // live-row windows differ by one activation row, into the same operand - when the lanes, the accumulator columns,
    // the per-thread work lists and shared memory allow it
    size_t fixed = 0;
    bool ok = false;
    for (p.S = 2; p.S >= 1 && !ok; --p.S) {
        if (p.S * 2 * p.KP > 128 || kNB * (g.AY + p.S - 1) > 256) continue;
        p.NP = 2 * p.S;
        p.nraw = ceil_div(p.NP * g.C * p.RW, kWorkers);
        p.nchunk = ceil_div(p.NP * p.KP * (kCT / 4), kWorkers);
        if (p.nraw > kRawMax || p.nchunk > kChunkMax) continue;
        p.stage_floats = p.NP * p.KP * kCT;
        // ring slots: AY + S at least; more while two operand stages still fit - a longer ring splits fewer live-row
        // windows at its wrap-around, and every split costs an extra MMA on the 46-clk issue floor
        for (p.RS = kRingMax; p.RS >= g.AY + p.S; --p.RS) {
            p.NRr = p.RS * kNB;
            p.ring_floats = (p.NRr * 4 + 4) * (kCT / 4);    // K-chunk stride padded by 16 bytes: conflict-free row staging
            fixed = (size_t)2 * p.ring_floats * 4 + (size_t)4 * p.NP * p.raw_floats * 4 + 4096;   // + over-read pad
            if (fixed + 2 * (size_t)2 * p.stage_floats * 4 <= (size_t)kMaxSmem) { ok = true; break; }
        }
        if (ok) break;
    }
    if (!ok) return false;
    p.n_stages = (int)(((size_t)kMaxSmem - fixed) / ((size_t)2 * p.stage_floats * 4));
    if (p.n_stages > kMaxStages) p.n_stages = kMaxStages;
    p.smem = fixed + (size_t)p.n_stages * 2 * p.stage_floats * 4;
    const long long cols = (long long)g.N * p.TXP;
    if (cols <= 0 || cols >= (1ll << 31) - kCT) return false;
    p.tiles = (int)((cols + kCT - 1) / kCT);
    const int sms = tma::sm_count();
    double best = -1;
    for (int rb = 1; rb <= g.TY && rb <= 64; ++rb) {
        const int rows = ceil_div(g.TY, rb);
        if (ceil_div(g.TY, rows) != rb) continue;
        const long long units = (long long)p.tiles * rb;
        const double waves = (double)((units + sms - 1) / sms);
        const double cost = waves * (rows + 0.5 * (g.AY - 1) + 1.0);
        if (best < 0 || cost < best * 0.999) { best = cost; p.rblocks = rb; p.rows_per_block = rows; }
    }
    p.units = (long long)p.tiles * p.rblocks;
    p.grid = (int)(p.units < sms ? p.units : sms);
    return true;
}

struct Unit {
    int tile, ty0, ty1, r_lo, r_hi;
};
__device__ __forceinline__ Unit make_unit(long long u, const Geo2 &g, const Plan &p) {
    Unit w;
    const int rb = (int)(u / p.tiles);
    w.tile = (int)(u - (long long)rb * p.tiles);
    w.ty0 = rb * p.rows_per_block;
    w.ty1 = min(g.TY, w.ty0 + p.rows_per_block);
    w.r_lo = max(0, w.ty0 - g.offy);
    w.r_hi = min(g.DY - 1, w.ty1 - 1 - g.offy + g.AY - 1);
    return w;
}

__global__ void __launch_bounds__(kThreads, 1) gradw_tc_kernel(const Geo2 g, const Plan p, const Args a) {
    extern __shared__ __align__(128) float smem[];
    __shared__ __align__(8) unsigned long long a_full[kMaxStages], a_empty[kMaxStages], h_full[kRingMax], h_free[kRingMax], set_done[2],
        set_free[2];
    __shared__ unsigned tmem_base_s;
    __shared__ __align__(16) int koff[64];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int KP = p.KP, AY = g.AY, AX = g.AX, C = g.C, RS = p.RS, RW = p.RW, S = p.S, NP = p.NP;
    float *ring_hi = smem, *ring_lo = smem + p.ring_floats;
    float *raw = ring_lo + p.ring_floats;                       // [2 buffers][hi, lo][plane][raw_floats]
    float *stages = raw + 4 * NP * p.raw_floats;                     // [stage][hi, lo][stage_floats]

    if (tid == 0) {
        for (int s = 0; s < p.n_stages; ++s) { mbar_init(&a_full[s], kWorkers); mbar_init(&a_empty[s], kIssuers); }
        for (int s = 0; s < kRingMax; ++s) { mbar_init(&h_full[s], kWorkers); mbar_init(&h_free[s], kIssuers); }
        for (int s = 0; s < 2; ++s) { mbar_init(&set_done[s], kIssuers); mbar_init(&set_free[s], 128); }
        mbar_fence_init();
    }
    if (warp == 8) tmem_alloc(&tmem_base_s, 512);
    if (tid < KP) koff[tid] = tid < C * AX ? (tid / AX) * RW + (tid % AX) : C * RW;
    // zeros behind every raw array (read through the padded k) - written once
    for (int idx = tid; idx < 4 * NP * (kCT + 8); idx += kThreads)
        raw[(idx / (kCT + 8)) * p.raw_floats + C * RW + (idx % (kCT + 8))] = 0.f;
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const unsigned tmem_base = tmem_base_s;
    if (warp < 4) {                                             // accumulator = 0
        for (int c = 0; c < 512; c += 16) tmem_st16_zero(tmem_base + ((unsigned)(warp * 32) << 16) + (unsigned)c);
        tmem_st_wait();
    }
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();

    const long long count = (long long)g.M * C * a.AYW * AX;

    if (warp < 8) {
        // ------------------------------------ workers ------------------------------------
        int st = 0;
        unsigned ph = 0, buf = 0;
        TC_PROF_DECL(empty); TC_PROF_DECL(hfree); TC_PROF_DECL(bar); TC_PROF_DECL(total); TC_PROF_DECL(hst); TC_PROF_DECL(rawp); TC_PROF_DECL(exp);
#ifdef TNMF_TC_PROFILE
        prof_total = -clock64();
#endif
        const long long plane = (long long)g.DY * g.DX;
        const int raw_count = NP * C * RW;
        // operand chunks of this thread: q = tid + 256 e -> (column group cg, operand row); fixed for the kernel
        int c_src[kChunkMax], c_dst[kChunkMax];
#pragma unroll
        for (int e = 0; e < kChunkMax; ++e) {
            const int q = tid + kWorkers * e;
            c_src[e] = -1;
            c_dst[e] = 0;
            if (e < p.nchunk && q < NP * KP * (kCT / 4)) {
                const int cg = q / (NP * KP), row = q - cg * (NP * KP);
                const int P = row / KP, k = row - P * KP;            // plane = (source row s, V | R)
                c_src[e] = P * p.raw_floats + koff[k] + 4 * cg;
                c_dst[e] = (row >> 3) * 32 + cg * (NP * KP * 4) + (row & 7) * 4;
            }
        }
        // activation chunk of this thread: atom ml, columns 4 cg .. 4 cg + 3 of the tile
        const int h_ml = tid >> 4, h_cg = tid & 15;
        long long g_base = 0;
        for (long long u = blockIdx.x; u < p.units; u += gridDim.x) {
            const Unit w = make_unit(u, g, p);
            // source element of every raw slot (q = tid + 256 e -> tensor, channel, position) in row 0, or -1: zero
            long long roff[kRawMax];
#pragma unroll
            for (int e = 0; e < kRawMax; ++e) {
                roff[e] = -1;
                const int q = tid + kWorkers * e;
                if (e < p.nraw && q < raw_count) {
                    const int qq = q % (C * RW);
                    const int c = qq / RW;
                    const long long J = (long long)w.tile * kCT + (qq - c * RW);
                    const int n = (int)(J / p.TXP);
                    const int x = (int)(J - (long long)n * p.TXP) - g.offx;
                    if (n < g.N && (unsigned)x < (unsigned)g.DX) roff[e] = ((long long)n * C + c) * plane + x;
                }
            }
            // activations: element offsets of the 4 columns in row 0 of atom m0 + ml, or -1: zero (gap column, no atom)
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
                    const int P = (tid + kWorkers * e) / (C * RW);       // plane -> source row r + P / 2, tensor P & 1
                    const int rr = r + (P >> 1);
                    const float *src = (P & 1) ? a.R : a.V;
                    rv[e] = (roff[e] >= 0 && rr <= w.r_hi) ? __ldg(src + (long long)rr * g.DX + roff[e]) : 0.f;
                }
            };
            // activation row fetch, issued one source row ahead of its use (interior rows bring exactly one new row)
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
            for (int r = w.r_lo; r <= w.r_hi; r += S) {
                // ---- activation rows that enter the window with this group of source rows ----
                const int t_b = min(w.ty1 - 1, min(r + S - 1, w.r_hi) + g.offy);
                unsigned new_slots = 0;
                for (; next_new <= t_b; ++next_new) {
                    const long long gi = g_base + (next_new - w.ty0);
                    const int slot = (int)(gi % RS);
                    const float4 hv = next_new == hv_row ? hv_next : load_h(next_new);
                    if (gi >= RS) TC_PROF_WAIT(hfree, mbar_wait_backoff(&h_free[slot], (unsigned)(((gi / RS) - 1) & 1), 40));
#ifdef TNMF_TC_PROFILE
                    const long long t_h = clock64();
#endif
                    float4 hi, lo;
                    split_tf32(hv.x, hi.x, lo.x); split_tf32(hv.y, hi.y, lo.y);
                    split_tf32(hv.z, hi.z, lo.z); split_tf32(hv.w, hi.w, lo.w);
                    const int nrow = slot * kNB + h_ml;
                    const size_t o = (size_t)(nrow >> 3) * 32 + (size_t)h_cg * (p.NRr * 4 + 4) + (size_t)(nrow & 7) * 4;
                    *reinterpret_cast<float4 *>(ring_hi + o) = hi;
                    *reinterpret_cast<float4 *>(ring_lo + o) = lo;
                    new_slots |= 1u << slot;                            // published below, behind one proxy fence
#ifdef TNMF_TC_PROFILE
                    prof_hst += clock64() - t_h;
#endif
                }
#ifdef TNMF_TC_PROFILE
                const long long t_r = clock64();
#endif
                // ---- expanded V and R rows ----
                float *raw_hi = raw + (size_t)buf * 2 * NP * p.raw_floats, *raw_lo = raw_hi + NP * p.raw_floats;
#pragma unroll
                for (int e = 0; e < kRawMax; ++e) {
                    const int q = tid + kWorkers * e;
                    if (e < p.nraw && q < raw_count) {
                        float hi, lo;
                        split_tf32(rv[e], hi, lo);
                        const int P = q / (C * RW);
                        raw_hi[P * p.raw_floats + (q - P * C * RW)] = hi;
                        raw_lo[P * p.raw_floats + (q - P * C * RW)] = lo;
                    }
                }
                if (r + S <= w.r_hi) load_raw(r + S);                 // in flight while this group is expanded
                if (next_new < w.ty1) { hv_next = load_h(next_new); hv_row = next_new; }
#ifdef TNMF_TC_PROFILE
                prof_rawp += clock64() - t_r;
#endif
                TC_PROF_WAIT(bar, asm volatile("bar.sync 1, 256;\n" ::: "memory"));
                TC_PROF_WAIT(empty, mbar_wait_backoff(&a_empty[st], ph ^ 1u, 40));
#ifdef TNMF_TC_PROFILE
                const long long t_e = clock64();
#endif
                float *d_hi = stages + (size_t)st * 2 * p.stage_floats, *d_lo = d_hi + p.stage_floats;
#pragma unroll
                for (int e = 0; e < kChunkMax; ++e) {
                    if (c_src[e] >= 0) {
                        const float *sh = raw_hi + c_src[e], *sl = raw_lo + c_src[e];
                        *reinterpret_cast<float4 *>(d_hi + c_dst[e]) = make_float4(sh[0], sh[1], sh[2], sh[3]);
                        *reinterpret_cast<float4 *>(d_lo + c_dst[e]) = make_float4(sl[0], sl[1], sl[2], sl[3]);
                    }
                }
                fence_proxy_async();
                for (; new_slots; new_slots &= new_slots - 1) mbar_arrive(&h_full[__ffs(new_slots) - 1]);
                mbar_arrive(&a_full[st]);
#ifdef TNMF_TC_PROFILE
                prof_exp += clock64() - t_e;
#endif
                if (++st == p.n_stages) { st = 0; ph ^= 1u; }
                buf ^= 1u;
            }
            g_base += w.ty1 - w.ty0;
        }
#ifdef TNMF_TC_PROFILE
        prof_total += clock64();
        if (blockIdx.x == 0 && tid == 0)
            printf("gradw workers: total %lld  wait a_empty %lld  wait h_free %lld  raw barrier %lld  h staging %lld  raw %lld  "
                   "expansion %lld\n", prof_total, prof_empty, prof_hfree, prof_bar, prof_hst, prof_rawp, prof_exp);
#endif
    } else if (warp >= 8 + kIssuers) {
        // ------------------------------------ accumulator drainers ------------------------------------
        // one accumulator set per epoch: lane = operand row k' = (X, c, ax), column = (ay, atom)
        long long rows_done = 0;
        bool first_drain = !a.accumulate;
        auto drain = [&](long long e) {
            const int set = (int)(e & 1);
            mbar_wait_backoff(&set_done[set], (unsigned)((e >> 1) & 1), 100);
            tc_fence_after();
            const int l = (warp & 3) * 32 + lane;
            const int P = l / KP, k = l - P * KP;                       // plane = (stacked row s, V | R)
            const int sr = P >> 1, X = P & 1;
            const bool live = P < NP && k < C * AX;
            const int c = live ? k / AX : 0, ax = live ? k - c * AX : 0;
            float *slice = a.partials + ((long long)blockIdx.x * S + sr) * 2 * count + (long long)X * count;
            const unsigned tbase = tmem_base + ((unsigned)((warp & 3) * 32) << 16) + (unsigned)(set * 256);
            for (int j = 0; j < AY + S - 1; ++j) {
                float v[16];
                tmem_ld16(tbase + (unsigned)(j * kNB), v);
                tmem_ld_wait();
                tmem_st16_zero(tbase + (unsigned)(j * kNB));
                const int ay = AY - 1 - j + sr;                         // stacked row s sees the window one row later
                if (live && ay >= 0 && ay < AY) {
                    // all 16 running sums are fetched before the first store (stores would otherwise order the loads)
                    float *dst0 = slice + (((long long)a.m0 * C + c) * a.AYW + a.ay0 + ay) * AX + ax;
                    const long long mstride = (long long)C * a.AYW * AX;
                    float old[kNB];
#pragma unroll
                    for (int ml = 0; ml < kNB; ++ml)
                        old[ml] = (!first_drain && a.m0 + ml < g.M) ? __ldcg(dst0 + ml * mstride) : 0.f;
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
            rows_done += (w.r_hi - w.r_lo + S) / S;                 // groups of S source rows
        }
        const long long n_epochs = (rows_done + kEpoch - 1) / kEpoch;
        for (long long e = 0; e < n_epochs; ++e) drain(e);
    } else {
        // ------------------------------------ MMA issuers (converged warps, one elected lane each) ------------------------------------
        const unsigned lbo_a = (unsigned)(NP * KP) * 16, lbo_b = (unsigned)p.NRr * 16 + 16;   // ring chunks carry a 16-byte pad
        const unsigned desc_hi = (128u >> 4) | (1u << 14);                      // SBO, descriptor version 1
        const unsigned a_lo_word = ((lbo_a >> 4) << 16), b_lo_word = ((lbo_b >> 4) << 16);
        const unsigned ring16[3] = {smem_u32(ring_hi) >> 4, smem_u32(ring_hi) >> 4, smem_u32(ring_lo) >> 4};
        const unsigned stage_addr0 = smem_u32(stages);
        const unsigned a_step16 = (2 * lbo_a) >> 4, b_step16 = (2 * lbo_b) >> 4;
        const int x = warp - 8;                 // warp 8 issues the first run of the live-row window, warp 9 the second
        int st = 0;
        unsigned ph = 0;
        long long g_base = 0, rows_done = 0;
        TC_PROF_DECL(full); TC_PROF_DECL(hfull); TC_PROF_DECL(setfree); TC_PROF_DECL(total);
#ifdef TNMF_TC_PROFILE
        prof_total = -clock64();
#endif
        for (long long u = blockIdx.x; u < p.units; u += gridDim.x) {
            const Unit w = make_unit(u, g, p);
            int next_new = w.ty0, next_out = w.ty0;
            for (int r = w.r_lo; r <= w.r_hi; r += S) {
                const int r_end = min(r + S - 1, w.r_hi);           // last source row of the group
                const long long epoch = rows_done / kEpoch;
                if (rows_done % kEpoch == 0 && epoch >= 2) {
                    TC_PROF_WAIT(setfree, mbar_wait(&set_free[epoch & 1], (unsigned)(((epoch >> 1) - 1) & 1)));
                    tc_fence_after();
                }
                const unsigned tset = tmem_base + (unsigned)((epoch & 1) * 256);
                const int ay_hi = min(AY - 1, r + g.offy - w.ty0);
                const int t_a = r + g.offy - ay_hi, t_b = min(w.ty1 - 1, r_end + g.offy);
                const int j0 = r + g.offy - AY + 1;                 // activation row of accumulator column block 0
                for (; next_new <= t_b; ++next_new) {
                    const long long gi = g_base + (next_new - w.ty0);
                    TC_PROF_WAIT(hfull, mbar_wait(&h_full[gi % RS], (unsigned)((gi / RS) & 1)));
                }
                TC_PROF_WAIT(full, mbar_wait(&a_full[st], ph));
                tc_fence_after();
                // The window [t_a, t_b] is cut into kIssuers runs of ring slots, one per issuing warp: at the ring's
                // wrap-around when it wraps, else in the middle.  Each warp issues ALL K steps of its run, so the runs
                // accumulate into disjoint TMEM columns in a fixed order - the result does not depend on how the two
                // warps interleave in the tensor pipe (splitting the K steps between the warps did: bitwise
                // run-to-run differences, caught by the graph-vs-eager test).
                const unsigned a_hi16 = (stage_addr0 + (unsigned)st * 2u * (unsigned)p.stage_floats * 4u) >> 4;
                const unsigned a_addr16[3] = {a_hi16, a_hi16 + (((unsigned)p.stage_floats * 4u) >> 4), a_hi16};
                auto issue_run = [&](unsigned o_col, unsigned o_idesc, unsigned o_b16) {
                    for (int ks = 0; ks < kCT / 8; ++ks) {
#pragma unroll
                        for (int t = 0; t < 3; ++t) {
                            const unsigned long long da =
                                ((unsigned long long)desc_hi << 32) | (a_lo_word | (a_addr16[t] + ks * a_step16));
                            const unsigned b16 = ring16[t] + ks * b_step16;
                            mma_tf32_elect(tset + o_col, da,
                                           ((unsigned long long)desc_hi << 32) | (b_lo_word | (b16 + o_b16)), o_idesc, 1u);
                        }
                    }
                };
                {
                    const int cnt = t_b - t_a + 1;
                    const int s0 = (int)((g_base + (t_a - w.ty0)) % RS);
                    int first = min(cnt, RS - s0);                      // slots before the wrap-around
                    if (kIssuers > 1 && first == cnt && cnt > 1) first = (cnt + 1) / 2;
                    if (kIssuers == 1 || x == 0)
                        issue_run((unsigned)((t_a - j0) * kNB), idesc_tf32(128, kNB * first), (unsigned)s0 * 16u);
                    if ((kIssuers == 1 || x == 1) && cnt > first)
                        issue_run((unsigned)((t_a - j0 + first) * kNB), idesc_tf32(128, kNB * (cnt - first)),
                                  (unsigned)((s0 + first) % RS) * 16u);
                }
                mma_commit_elect(&a_empty[st]);
                if (++st == p.n_stages) { st = 0; ph ^= 1u; }
                // activation rows that leave the window: their slots may be overwritten once these MMAs are done
                for (; next_out < w.ty1 && min(g.DY - 1, next_out - g.offy + AY - 1) <= r_end; ++next_out)
                    mma_commit_elect(&h_free[(g_base + (next_out - w.ty0)) % RS]);
                if (++rows_done % kEpoch == 0) mma_commit_elect(&set_done[epoch & 1]);
            }
            g_base += w.ty1 - w.ty0;
        }
        if (rows_done % kEpoch != 0) mma_commit_elect(&set_done[(rows_done / kEpoch) & 1]);
#ifdef TNMF_TC_PROFILE
        prof_total += clock64();
        if (blockIdx.x == 0 && lane == 0 && x == 0)
            printf("gradw mma: total %lld  wait a_full %lld  wait h_full %lld  wait set_free %lld\n", prof_total, prof_full,
                   prof_hfull, prof_setfree);
#endif
        __syncwarp();
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 8) tmem_dealloc(tmem_base, 512);
}

}  // namespace gw
}  // namespace tc

// ---- dispatch ----------------------------------------------------------------------------------------------------------
// Tall atoms (A_y > 15, 'valid' mode): rows [a0, a0 + h) of the W gradient are the W gradient of an h-row atom against H
// moved down by A_y - a0 - h rows (H row = d_y + (A_y - 1) - a_y = d_y + (h - 1 - a') + (A_y - a0 - h)), so the atom is cut
// into row chunks that the kernel above serves one after the other.  All chunks add into the same zeroed per-CTA slices
// (disjoint entries), and one fixed-order finish sums them: still deterministic, no atomics.
namespace tc {
namespace gw {
static Geo2 chunk_geo(const Geo2 &q, int h) {
    Geo2 s = q;
    s.AY = h; s.TY = q.DY + h - 1; s.offy = h - 1;
    return s;
}
static bool plan_tall(const Geo2 &q, int &h, int &n) {
    if (q.AY <= 15 || q.wrap || q.offy != q.AY - 1 || q.TY != q.DY + q.AY - 1) return false;
    Plan p;
    for (h = 15; h >= 2; --h)
        if (make_plan(chunk_geo(q, h), p)) break;
    if (h < 2) return false;
    n = ceil_div(q.AY, h);
    h = ceil_div(q.AY, n);                                      // balanced chunks; the last one may be shorter
    for (int a0 = 0; a0 < q.AY; a0 += h)
        if (!make_plan(chunk_geo(q, q.AY - a0 < h ? q.AY - a0 : h), p)) return false;
    return true;
}
}  // namespace gw
}  // namespace tc

bool tc_gradw_supported(const Geo &g, int dtype) {
    if (!tc::rank2_ok(g, dtype)) return false;
    tc::gw::Plan p;
    const tiled::Geo2 q = tiled::make_geo2(g);
    int h, n;
    return tc::gw::make_plan(q, p) || tc::gw::plan_tall(q, h, n);
}

size_t tc_gradw_workspace_bytes(const Geo &g) {
    tc::gw::Plan p;
    const tiled::Geo2 q = tiled::make_geo2(g);
    const size_t slice = 2 * (size_t)g.M * g.C * g.A[1] * g.A[2] * sizeof(float);
    if (tc::gw::make_plan(q, p)) return (size_t)p.grid * p.S * slice;
    int h, n;
    if (tc::gw::plan_tall(q, h, n)) return (size_t)tma::sm_count() * 2 * slice;     // any grid, any stacking
    return 0;
}

int tc_gradient_w(const Geo &g, const float *V, const float *R, const float *H, float *neg, float *pos, void *workspace,
                  size_t workspace_bytes, cudaStream_t st) {
    const tiled::Geo2 q = tiled::make_geo2(g);
    tc::gw::Plan p;
    int h = 0, n = 0;
    const bool whole = tc::gw::make_plan(q, p);
    if (!whole && !tc::gw::plan_tall(q, h, n)) return TNMF_EUNSUPPORTED;
    const long long count = (long long)g.M * g.C * g.A[1] * g.A[2];
    if (!workspace || workspace_bytes < tc_gradw_workspace_bytes(g)) return TNMF_EWORKSPACE;
    cudaError_t e = cudaFuncSetAttribute(tc::gw::gradw_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         tc::gw::kMaxSmem);
    if (e != cudaSuccess) return status_from_cuda(e);
    tc::gw::Args a;
    a.V = V; a.R = R; a.H = H; a.partials = (float *)workspace;
    a.ay0 = 0; a.AYW = q.AY; a.accumulate = 0;
    if (whole) {
        for (int m0 = 0; m0 < g.M; m0 += tc::gw::kNB) {
            a.m0 = m0;
            tc::gw::gradw_tc_kernel<<<(unsigned)p.grid, tc::gw::kThreads, p.smem, st>>>(q, p, a);
            TNMF_CHECK_LAUNCH();
        }
        return finish_gradient_w<float>((const float *)workspace, p.grid * p.S, count, neg, pos, st);
    }
    const int slices = tma::sm_count() * 2;
    e = cudaMemsetAsync(workspace, 0, (size_t)slices * 2 * count * sizeof(float), st);
    if (e != cudaSuccess) return status_from_cuda(e);
    a.accumulate = 1;
    for (int a0 = 0; a0 < q.AY; a0 += h) {
        const int hc = q.AY - a0 < h ? q.AY - a0 : h;
        const tiled::Geo2 sub = tc::gw::chunk_geo(q, hc);
        if (!tc::gw::make_plan(sub, p)) return TNMF_EUNSUPPORTED;
        a.ay0 = a0;
        a.H = H + (long long)(q.AY - a0 - hc) * q.hsy;
        for (int m0 = 0; m0 < g.M; m0 += tc::gw::kNB) {
            a.m0 = m0;
            tc::gw::gradw_tc_kernel<<<(unsigned)p.grid, tc::gw::kThreads, p.smem, st>>>(sub, p, a);
            TNMF_CHECK_LAUNCH();
        }
    }
    return finish_gradient_w<float>((const float *)workspace, slices, count, neg, pos, st);
}

int tc_gradw_launches(const Geo &g) {
    const tiled::Geo2 q = tiled::make_geo2(g);
    tc::gw::Plan p;
    int h = 0, n = 1;
    if (!tc::gw::make_plan(q, p)) tc::gw::plan_tall(q, h, n);
    return n * tiled::ceil_div(g.M, tc::gw::kNB) + 1;
}

}  // namespace tnmf
