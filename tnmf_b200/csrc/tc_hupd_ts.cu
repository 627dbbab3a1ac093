// Tensor-core (tcgen05, 3xTF32) H gradient with the fused multiplicative update, expanded operand in TENSOR MEMORY.
//
//   neg[n,m,ty,tx] = sum_c sum_{ay,ax} W[m,c,ay,ax] * Vext[n,c,ty-offy+ay,tx-offx+ax]   (tnmf/backends/NumPy.py:101-109)
//   pos[n,m,ty,tx] = the same with R                                                    (tnmf/backends/NumPy.py:111-119)
//   epilogue (H given):  pos += lambda*(G-H); pos += lambda_c*(Gsum-G); pos += reg; H = (H*neg)/pos
//                                                           (tnmf/TransformInvariantNMF.py:217-235,246-271)
//
// Same product as tc_hupd.cu: a CTA owns 128 activation COLUMNS (column J = n * TXP + xv of the flattened [N x TXP] space,
// TXP = TX + AX - 1) and walks down the source rows; for a source row r of X (V or R)
//       A_r[column i, k = (c, ax)] = Xext[n_i, c, r, tx_i - offx + ax]          D_ty[column, m] += A_r[column, :] . Wt_ay[m, :]
// for all output rows ty = r + offy - ay at once (N = 16 atoms x live rows, output rows in a ring of TMEM slots).  What
// changes is where A_r lives: in TENSOR MEMORY, lane = column, 32-bit TMEM column = k.  The thread that owns a column reads its
// C*AX-wide window of the raw source row (LDS.32, consecutive lanes consecutive words), splits hi/lo in registers and writes
// its lane with tcgen05.st.  The MMA then fetches only the atom operand from shared memory (the 4 KB A fetch per MMA was 40 %
// of the port's traffic), the expansion's STS.128 into 8-row core matrices is gone, and so is its bank-conflict rate.
//
// TMEM columns: neg ring (RS slots x 16 atoms), pos ring (the same), then one operand buffer per tensor (KP hi + KP lo
// columns each).  cfg2 (KP = 40, AY = 11): 176 + 176 + 160 = 512 with RS = AY, i.e. no spare slot - which works because a
// finished row is drained in two halves: neg after the V stage that completes it (while the R stage runs), pos after the
// R stage (while the next V stage runs).  The epilogue zeroes a slot when it has read it, so every MMA accumulates.
//
// Roles (576 threads): warps 0-3 expand V rows, warps 4-7 R rows (thread = column = TMEM lane); warp 8 issues the V stages
// (neg ring), warp 9 the R stages (pos ring) - converged warps, one election per stage, operands in uniform registers - and
// they take turns (V(r), R(r), V(r+1), ...: while one tensor's MMAs run, the other tensor's next row is expanded into its
// single operand buffer); warps 10-17 run the epilogue (two warps per TMEM lane quarter, eight atoms each).  mbarriers: a_full/a_empty per tensor, {neg,pos}_{done,free} per
// ring slot, turn per issuer.  Atoms in blocks of 16 (one launch per block).
#include "tc_common.cuh"

namespace tnmf {
namespace tc {
namespace hut {

using tiled::ceil_div;
using tiled::Geo2;
using tiled::round_up;

constexpr int kTile = 128;          // activation columns per CTA tile = MMA M
constexpr int kNB = 16;             // atoms per launch
constexpr int kThreads = 32 * 18;     // 8 expander + 2 MMA-issuing + 8 epilogue warps
constexpr int kRingMax = 16;
constexpr int kRawMax = 8;          // raw-row elements per expander thread (C * (128 + AX - 1) <= 1024)
constexpr int kMaxSmem = 226 * 1024;

struct Plan {
    int KPL, KP, ksteps;            // C*AX, padded to a multiple of 8
    int TXP, RW, raw_floats, nraw;
    int RS, pos_col0, a_col0;       // ring slots, first TMEM column of the pos ring / of the operand buffers
    int shared_ab;                  // 1: V and R take turns in ONE operand buffer (the rings leave room for one only)
    int w_floats;
    int tiles;
    long long total, quota, units;  // tile-rows of the problem, tile-rows per CTA, grid * (most segments of a CTA)
    int grid;
    size_t smem;
    int koff[64];                   // k = (c, ax) -> c * RW + ax: offset of the tap in a raw row (kernel parameters live in
                                    // the constant bank: the expanders add them as immediate-like operands)
};

struct Args {
    const float *V, *R, *W;
    float *neg, *pos, *H;
    float reg, lambda, lambda_cross;
    const float *G, *Gsum;
    int m0;
};

bool make_plan(const Geo2 &g, Plan &p) {
    p = Plan();
    if (g.AY < 1) return false;
    p.KPL = g.C * g.AX;
    if (p.KPL > 64) return false;
    p.KP = round_up(p.KPL, 8);
    p.ksteps = p.KP / 8;
    p.RS = (512 - 4 * p.KP) / (2 * kNB);
    if (p.RS > kRingMax) p.RS = kRingMax;
    if (p.RS < g.AY) {
        // one operand buffer for both tensors (cfg3: 15 atom rows -> 480 ring columns + 2 * KP = 512): the V and R stages
        // alternate anyway; what is lost is the expansion of one tensor running under the other tensor's MMAs
        p.RS = (512 - 2 * p.KP) / (2 * kNB);
        if (p.RS > kRingMax) p.RS = kRingMax;
        if (p.RS < g.AY) return false;
        p.shared_ab = 1;
    }
    p.pos_col0 = p.RS * kNB;
    p.a_col0 = 2 * p.RS * kNB;
    p.w_floats = 2 * g.AY * kNB * p.KP;
    p.TXP = g.TX + g.AX - 1;
    p.RW = kTile + g.AX - 1;
    p.raw_floats = round_up(g.C * p.RW, 32);
    p.nraw = ceil_div(g.C * p.RW, 128);
    if (p.nraw > kRawMax) return false;
    for (int k = 0; k < 64; ++k) p.koff[k] = k < p.KPL ? (k / g.AX) * p.RW + (k % g.AX) : 0;
    p.smem = (size_t)p.w_floats * 4 + (size_t)4 * p.raw_floats * 4 + 1024;
    if (p.smem > (size_t)kMaxSmem) return false;
    const long long cols = (long long)g.N * p.TXP;
    if (cols <= 0 || cols >= (1ll << 31) - kTile) return false;
    p.tiles = (int)((cols + kTile - 1) / kTile);
    // Work split: the (tile, row) space is cut into `grid` equal LINEAR ranges, one per CTA (a range is a few row segments
    // of consecutive tiles) - every SM gets the same number of rows whatever the number of tiles (cfg2: 138 / 145 / 276
    // tiles on 148 SMs left 7 - 10 % of the SMs idle with whole-tile units).  A segment boundary costs AY - 1 extra source
    // rows, and there are at most two per CTA.
    const int sms = tma::sm_count();
    p.total = (long long)p.tiles * g.TY;
    p.quota = (p.total + sms - 1) / sms;
    const long long min_quota = g.TY < 8 ? g.TY : 8;
    if (p.quota < min_quota) p.quota = min_quota;
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
    const long long lo = b * p.quota, hi = min(lo + p.quota, p.total);
    w.tile = (int)(lo / g.TY + k);
    const long long t0 = (long long)w.tile * g.TY;
    const long long s0 = max(lo, t0), s1 = min(hi, t0 + g.TY);
    w.ty0 = s1 > s0 ? (int)(s0 - t0) : 0;
    w.ty1 = s1 > s0 ? (int)(s1 - t0) : 0;
    w.r_lo = max(0, w.ty0 - g.offy);
    w.r_hi = min(g.DY - 1, w.ty1 - 1 - g.offy + g.AY - 1);
    return w;
}

// KPT = KP: compile-time contraction length (the expansion is fully unrolled: all loads of a row in flight at once);
// P3: plane mode (G = Geo3, tc_common.cuh) - virtual samples (n, t_z), virtual channels (c, a_z) reading source plane
// t_z - offz + a_z, or zeros outside [0, D_z)
template <int KPT, bool P3, class G>
__device__ __forceinline__ void hupd_ts_body(const G &g, const Plan &p, const Args &a) {
    extern __shared__ __align__(128) float smem[];
    __shared__ __align__(8) unsigned long long a_full[2], a_empty[2], turn[2], x_done[2][kRingMax], x_free[2][kRingMax];
    __shared__ unsigned tmem_base_s;
    const int tid = threadIdx.x, warp = __shfl_sync(0xffffffffu, tid >> 5, 0), lane = tid & 31;
    const int KP = p.KP, AY = g.AY, AX = g.AX, C = g.C, RS = p.RS, RW = p.RW;
    const int NR = AY * kNB;                                // rows of the atom operand
    float *w_hi = smem, *w_lo = smem + NR * KP;
    float *raw = smem + p.w_floats;                         // [tensor][2 buffers][raw_floats]

    if (tid == 0) {
        for (int s = 0; s < 2; ++s) { mbar_init(&a_full[s], 4); mbar_init(&a_empty[s], 1); mbar_init(&turn[s], 1); }
        for (int x = 0; x < 2; ++x)
            for (int s = 0; s < kRingMax; ++s) { mbar_init(&x_done[x][s], 1); mbar_init(&x_free[x][s], 8); }
        mbar_fence_init();
    }
    if (warp == 8) tmem_alloc(&tmem_base_s, 512);
    // atom operand: row n = j*16 + ml  <->  atom m0+ml, atom row ay = AY-1-j;  k = c*AX + ax
    for (int idx = tid; idx < NR * KP; idx += kThreads) {
        const int n = idx / KP, k = idx - n * KP;
        const int j = n / kNB, ml = n - j * kNB;
        const int m = a.m0 + ml, ay = AY - 1 - j;
        float v = 0.f;
        if (m < g.M && k < p.KPL) {
            const int c = k / AX, ax = k - c * AX;
            v = a.W[(((long long)m * C + c) * AY + ay) * AX + ax];
        }
        float hi, lo;
        split_tf32(v, hi, lo);
        const size_t o = canon_offset_floats(n, k, NR);
        w_hi[o] = hi;
        w_lo[o] = lo;
    }
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const unsigned tmem_base = tmem_base_s;
    if (warp < 4) {                                             // rings = 0 (every MMA accumulates), operand pads = 0
        for (int c = 0; c < 512; c += 16) tmem_st16_zero(tmem_base + ((unsigned)(warp * 32) << 16) + (unsigned)c);
        tmem_st_wait();
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();

    if (warp < 8) {
        // ------------------------------------ expanders: X = 0 (V) warps 0-3, X = 1 (R) warps 4-7 ------------------------------------
        const int X = warp >> 2, quarter = warp & 3;
        const int i = quarter * 32 + lane;                      // column of the tile = TMEM lane
        const int t128 = tid & 127;
        const float *src_t = X ? a.R : a.V;
        float *raw_x = raw + (size_t)X * 2 * p.raw_floats;
        const unsigned t_lane = tmem_base + ((unsigned)(quarter * 32) << 16) +
                                (unsigned)(p.a_col0 + (p.shared_ab ? 0 : X * 2 * KP));
        const long long plane = (long long)g.DY * g.DX;
        const int raw_count = C * RW;
        unsigned stage = 0, buf = 0;
        TC_PROF_DECL(empty); TC_PROF_DECL(total); TC_PROF_DECL(bar); TC_PROF_DECL(exp);
#ifdef TNMF_TC_PROFILE
        prof_total = -clock64();
#endif
        for (long long u = blockIdx.x; u < p.units; u += gridDim.x) {
            const Unit w = make_unit(u, g, p);
            if (w.ty0 >= w.ty1) break;                            // past this CTA's last segment
            // source element of every raw slot (q = t128 + 128 e -> channel q / RW, position q % RW) in row 0, or -1: zero
            long long roff[kRawMax];
#pragma unroll
            for (int e = 0; e < kRawMax; ++e) {
                roff[e] = -1;
                const int q = t128 + 128 * e;
                if (e < p.nraw && q < raw_count) {
                    const int c = q / RW;
                    const long long J = (long long)w.tile * kTile + (q - c * RW);
                    const int n = (int)(J / p.TXP);
                    const int x = (int)(J - (long long)n * p.TXP) - g.offx;
                    if (n < g.N && (unsigned)x < (unsigned)g.DX) {
                        if constexpr (P3) {
                            const int ns = n / g.NZ, cr = c / g.AZ, z = g.z0 + n - ns * g.NZ - g.offz + (c - cr * g.AZ);
                            if ((unsigned)z < (unsigned)g.DZ) roff[e] = ns * g.xsn + cr * g.xsc + (long long)z * plane + x;
                        } else {
                            roff[e] = ((long long)n * C + c) * plane + x;
                        }
                    }
                }
            }
            float rv[kRawMax];
            auto load_raw = [&](int r) {
                const float *src = src_t + (long long)r * g.DX;
#pragma unroll
                for (int e = 0; e < kRawMax; ++e) rv[e] = roff[e] >= 0 ? __ldg(src + roff[e]) : 0.f;
            };
            load_raw(w.r_lo);
            for (int r = w.r_lo; r <= w.r_hi; ++r, ++stage) {
                float *rb = raw_x + (size_t)buf * p.raw_floats;
#pragma unroll
                for (int e = 0; e < kRawMax; ++e)
                    if (e < p.nraw && t128 + 128 * e < raw_count) rb[t128 + 128 * e] = rv[e];
                if (r < w.r_hi) load_raw(r + 1);                    // in flight while this row is expanded and multiplied
                TC_PROF_WAIT(bar, asm volatile("bar.sync %0, 128;\n" ::"r"(1 + X) : "memory"));
                // window of this column: k = (c, ax) -> rb[c * RW + ax + i].  All loads are issued before the first use: under
                // the tensor core's operand traffic a shared-memory round trip costs ~150 clk (measured in tc_recon_ts.cu)
                const float *pw = rb + i;
                float v[KPT];
#pragma unroll
                for (int k = 0; k < KPT; ++k) v[k] = k < p.KPL ? pw[p.koff[k]] : 0.f;
                // the window is in registers before the operand buffer is free: only the split and the stores wait for it
                if (!p.shared_ab) {
                    if (stage) TC_PROF_WAIT(empty, mbar_wait_backoff(&a_empty[X], (stage - 1u) & 1u, 20));
                } else if (X) {
                    // one buffer, used in the order V(0) R(0) V(1) R(1) ...: R(s) may be written when the MMAs of V(s) are done
                    TC_PROF_WAIT(empty, mbar_wait_backoff(&a_empty[0], stage & 1u, 20));
                } else if (stage) {
                    TC_PROF_WAIT(empty, mbar_wait_backoff(&a_empty[1], (stage - 1u) & 1u, 20));     // V(s): after R(s - 1)
                }
                tc_fence_after();
#ifdef TNMF_TC_PROFILE
                const long long t_e = clock64();
#endif
#pragma unroll
                for (int k0 = 0; k0 < KPT; k0 += 16) {
                    if (k0 + 16 <= KPT) {
                        float hi[16], lo[16];
#pragma unroll
                        for (int j = 0; j < 16; ++j) split_tf32(v[k0 + j], hi[j], lo[j]);
                        tmem_st16(t_lane + (unsigned)k0, hi);
                        tmem_st16(t_lane + (unsigned)(KPT + k0), lo);
                    } else {                                        // KP is a multiple of 8: a tail of 8 columns
                        float h8[8], l8[8];
#pragma unroll
                        for (int j = 0; j < 8; ++j) split_tf32(v[k0 + j], h8[j], l8[j]);
                        tmem_st8(t_lane + (unsigned)k0, h8);
                        tmem_st8(t_lane + (unsigned)(KPT + k0), l8);
                    }
                }
                tmem_st_wait();
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(&a_full[X]);
#ifdef TNMF_TC_PROFILE
                prof_exp += clock64() - t_e;
#endif
                buf ^= 1u;
            }
        }
#ifdef TNMF_TC_PROFILE
        prof_total += clock64();
        if (blockIdx.x == 0 && (tid == 0 || tid == 128))
            printf("hupd_ts expanders X=%d: total %lld  wait a_empty %lld  raw barrier %lld  expansion %lld\n", X, prof_total, prof_empty, prof_bar, prof_exp);
#endif
    } else if (warp >= 10) {
        // ------------------------------------ epilogue: warps 10-13 atoms 0-7, warps 14-17 atoms 8-15 of the block ------------------------------------
        const int q = warp & 3, hs = (warp - 10) >> 2;
        constexpr int kHA = kNB / 2;
        const int i = q * 32 + lane;
        const unsigned lane_base = tmem_base + ((unsigned)(q * 32) << 16) + (unsigned)(hs * kHA);
        const int ma = a.m0 + hs * kHA;                        // first atom of this thread
        const long long tvol = (long long)g.TY * g.TX;
        int slot = 0;
        unsigned wraps = 0;
        TC_PROF_DECL(dneg); TC_PROF_DECL(dpos); TC_PROF_DECL(total);
#ifdef TNMF_TC_PROFILE
        prof_total = -clock64();
#endif
        for (long long u = blockIdx.x; u < p.units; u += gridDim.x) {
            const Unit w = make_unit(u, g, p);
            if (w.ty0 >= w.ty1) break;                            // past this CTA's last segment
            const long long J = (long long)w.tile * kTile + i;
            const int n = (int)(J / p.TXP);
            const int tx = (int)(J - (long long)n * p.TXP);
            const bool active = n < g.N && tx < g.TX;
            // the activations of a row do not depend on the accumulators: they are fetched one row ahead
            float hnext[kHA];
            long long hbase;
            if constexpr (P3) hbase = (long long)(n / g.NZ) * g.hsn + (long long)(g.z0 + n % g.NZ) * g.hsz;
            else hbase = (long long)n * g.hsn;
            float *hrow = (a.H && active) ? a.H + hbase + (long long)ma * g.hsm + tx : nullptr;
            auto load_h = [&](int ty) {
#pragma unroll
                for (int ml = 0; ml < kHA; ++ml)
                    hnext[ml] = (hrow && ma + ml < g.M) ? hrow[(long long)ty * g.hsy + (long long)ml * g.hsm] : 0.f;
            };
            const bool fast = a.H && !a.G && a.m0 + kNB <= g.M;
            load_h(w.ty0);
            for (int ty = w.ty0; ty < w.ty1; ++ty) {
                float neg[kHA], pos[kHA];
                // neg: final after the V stage of the row's last source row - drained while the R stage runs
                TC_PROF_WAIT(dneg, mbar_wait_backoff(&x_done[0][slot], wraps & 1u, 20));
                tc_fence_after();
                tmem_ld8(lane_base + (unsigned)(slot * kNB), neg);
                tmem_ld_wait();
                tmem_st8_zero(lane_base + (unsigned)(slot * kNB));
                tmem_st_wait();
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(&x_free[0][slot]);
                // pos: final after the R stage - drained while the next V stage runs
                TC_PROF_WAIT(dpos, mbar_wait_backoff(&x_done[1][slot], wraps & 1u, 20));
                tc_fence_after();
                tmem_ld8(lane_base + (unsigned)(p.pos_col0 + slot * kNB), pos);
                tmem_ld_wait();
                tmem_st8_zero(lane_base + (unsigned)(p.pos_col0 + slot * kNB));
                tmem_st_wait();
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(&x_free[1][slot]);
                if (++slot == RS) { slot = 0; ++wraps; }
                float hv[kHA];
#pragma unroll
                for (int ml = 0; ml < kHA; ++ml) hv[ml] = hnext[ml];
                if (fast) {
                    // plain fused update of a full block of 16 atoms: pointer walks, no per-atom tests.  The product and the
                    // quotient round separately and to nearest, like the reference's `arr *= neg; arr /= pos`.
                    if (active) {
                        float *o = hrow + (long long)ty * g.hsy;
                        if (ty + 1 < w.ty1) {
                            const float *qn = o + g.hsy;
#pragma unroll
                            for (int ml = 0; ml < kHA; ++ml) { hnext[ml] = *qn; qn += g.hsm; }
                        }
#pragma unroll
                        for (int ml = 0; ml < kHA; ++ml) {
                            *o = __fdiv_rn(__fmul_rn(hv[ml], neg[ml]), __fadd_rn(pos[ml], a.reg));
                            o += g.hsm;
                        }
                    }
                    continue;
                }
                if (ty + 1 < w.ty1) load_h(ty + 1);
                if (!active) continue;
                const long long tin = (long long)ty * g.TX + tx;
#pragma unroll
                for (int ml = 0; ml < kHA; ++ml) {
                    const int m = ma + ml;
                    if (m >= g.M) continue;
                    long long cidx;                 // dense [n][m][(t_z,) t_y][t_x] of the whole problem
                    if constexpr (P3) cidx = (((long long)(n / g.NZ) * g.M + m) * g.TZ + g.z0 + n % g.NZ) * tvol + tin;
                    else cidx = ((long long)n * g.M + m) * tvol + tin;
                    if (a.H) {
                        const float h = hv[ml];
                        float ps = pos[ml];
                        if (a.G) {
                            const float gv = a.G[cidx];
                            if (a.lambda != 0.f) { float tmp = gv - h; tmp *= a.lambda; ps += tmp; }
                            if (a.Gsum) {
                                long long sidx;         // Gsum: one atom
                                if constexpr (P3) sidx = ((long long)(n / g.NZ) * g.TZ + g.z0 + n % g.NZ) * tvol + tin;
                                else sidx = (long long)n * tvol + tin;
                                const float gs = a.Gsum[sidx];
                                float tmp = -gv + gs; tmp *= a.lambda_cross; ps += tmp;
                            }
                        }
                        ps += a.reg;
                        float hn = h * neg[ml];
                        hn /= ps;
                        hrow[(long long)ty * g.hsy + (long long)ml * g.hsm] = hn;
                    } else {
                        a.neg[cidx] = neg[ml];
                        a.pos[cidx] = pos[ml];
                    }
                }
            }
        }
#ifdef TNMF_TC_PROFILE
        prof_total += clock64();
        if (blockIdx.x == 0 && tid == 320) printf("hupd_ts epilogue: total %lld  wait neg_done %lld  wait pos_done %lld\n", prof_total, prof_dneg, prof_dpos);
#endif
    } else {
        // ------------------------------------ MMA issuers: warp 8 the V stages, warp 9 the R stages ------------------------------------
        const int X = warp - 8;
        const unsigned tmem_u = __shfl_sync(0xffffffffu, tmem_base, 0);
        const unsigned lbo_b = (unsigned)NR * 16;
        const unsigned desc_hi = (128u >> 4) | (1u << 14);      // SBO = 128, descriptor version 1
        const unsigned w_hi_word = __shfl_sync(0xffffffffu, (smem_u32(w_hi) >> 4) + ((lbo_b >> 4) << 16), 0);
        const unsigned w_lo_word = __shfl_sync(0xffffffffu, (smem_u32(w_lo) >> 4) + ((lbo_b >> 4) << 16), 0);
        const unsigned b_step16 = (2 * lbo_b) >> 4;
        const unsigned ring0 = tmem_u + (unsigned)(X ? p.pos_col0 : 0);
        const unsigned ta_hi = tmem_u + (unsigned)(p.a_col0 + (p.shared_ab ? 0 : X * 2 * KP)), ta_lo = ta_hi + (unsigned)KP;
        const int ksteps = p.ksteps;
        unsigned stage = 0;
        int slot_new = 0, slot_a = 0, slot_done = 0;            // slot of the next row to enter / of the window's first row /
        unsigned wraps_new = 0;                                 // of the next row to complete
        TC_PROF_DECL(xfree); TC_PROF_DECL(afull); TC_PROF_DECL(turnw); TC_PROF_DECL(issue); TC_PROF_DECL(total);
#ifdef TNMF_TC_PROFILE
        prof_total = -clock64();
#endif
        for (long long u = blockIdx.x; u < p.units; u += gridDim.x) {
            const Unit w = make_unit(u, g, p);
            if (w.ty0 >= w.ty1) break;                            // past this CTA's last segment
            int next_new = w.ty0, next_done = w.ty0, win0 = w.ty0;
            slot_a = slot_new;
            for (int r = w.r_lo; r <= w.r_hi; ++r, ++stage) {
                const int ay_lo = max(0, r + g.offy - (w.ty1 - 1)), ay_hi = min(AY - 1, r + g.offy - w.ty0);
                const int t_a = r + g.offy - ay_hi, t_b = r + g.offy - ay_lo;
                const int j0 = r + g.offy - AY + 1;                 // output row of atom-row block 0
                // output rows that receive their first contribution from this source row: their slot must have been drained
                for (; next_new <= t_b; ++next_new) {
                    if (wraps_new) TC_PROF_WAIT(xfree, mbar_wait(&x_free[X][slot_new], (wraps_new - 1u) & 1u));
                    if (++slot_new == RS) { slot_new = 0; ++wraps_new; }
                }
                for (; win0 < t_a; ++win0)
                    if (++slot_a == RS) slot_a = 0;
                TC_PROF_WAIT(afull, mbar_wait(&a_full[X], stage & 1u));
                // take turns with the other tensor's warp: V(r), R(r), V(r+1), ...
                if (X) TC_PROF_WAIT(turnw, mbar_wait(&turn[1], stage & 1u));
                else if (stage) TC_PROF_WAIT(turnw, mbar_wait(&turn[0], (stage - 1u) & 1u));
                tc_fence_after();
#ifdef TNMF_TC_PROFILE
                const long long t_i = clock64();
#endif
                // the live rows [t_a, t_b] are one run of ring slots, or two when the window wraps around the ring
                const int cnt = t_b - t_a + 1;
                const int first = min(cnt, RS - slot_a);
                const unsigned col0 = ring0 + (unsigned)(slot_a * kNB), idesc0 = idesc_tf32(kTile, kNB * first);
                const unsigned idesc1 = idesc_tf32(kTile, kNB * max(cnt - first, 1));
                const unsigned b0 = (unsigned)(t_a - j0) * 16u, b1 = b0 + (unsigned)first * 16u;
                const bool two = cnt > first;
                if (elect_one()) {
                    // compile-time K steps, the wrap branch outside the loop, the hand-over at a fixed step: between two MMAs
                    // the issuing lane executes uniform adds only
                    constexpr int kSteps = KPT / 8, kMid = (kSteps - 1) / 2;
                    if (two) {
#pragma unroll
                        for (int ks = 0; ks < kSteps; ++ks) {
                            const unsigned kb = (unsigned)ks * b_step16;
                            if (ks == kMid) mbar_arrive(&turn[X ^ 1]);              // half way: the other warp may start
                            mma_tf32_ts2<true>(col0, ta_hi + 8u * ks, w_hi_word + kb + b0, desc_hi, idesc0);
                            mma_tf32_ts2<true>(ring0, ta_hi + 8u * ks, w_hi_word + kb + b1, desc_hi, idesc1);
                            mma_tf32_ts2<true>(col0, ta_lo + 8u * ks, w_hi_word + kb + b0, desc_hi, idesc0);
                            mma_tf32_ts2<true>(ring0, ta_lo + 8u * ks, w_hi_word + kb + b1, desc_hi, idesc1);
                            mma_tf32_ts2<true>(col0, ta_hi + 8u * ks, w_lo_word + kb + b0, desc_hi, idesc0);
                            mma_tf32_ts2<true>(ring0, ta_hi + 8u * ks, w_lo_word + kb + b1, desc_hi, idesc1);
                        }
                    } else {
#pragma unroll
                        for (int ks = 0; ks < kSteps; ++ks) {
                            const unsigned kb = (unsigned)ks * b_step16;
                            if (ks == kMid) mbar_arrive(&turn[X ^ 1]);
                            mma_tf32_ts2<true>(col0, ta_hi + 8u * ks, w_hi_word + kb + b0, desc_hi, idesc0);
                            mma_tf32_ts2<true>(col0, ta_lo + 8u * ks, w_hi_word + kb + b0, desc_hi, idesc0);
                            mma_tf32_ts2<true>(col0, ta_hi + 8u * ks, w_lo_word + kb + b0, desc_hi, idesc0);
                        }
                    }
                }
                __syncwarp();
#ifdef TNMF_TC_PROFILE
                prof_issue += clock64() - t_i;
#endif
                mma_commit_elect(&a_empty[X]);
                // output rows whose last source row this was
                for (; next_done < w.ty1 && min(g.DY - 1, next_done - g.offy + AY - 1) <= r; ++next_done) {
                    mma_commit_elect(&x_done[X][slot_done]);
                    if (++slot_done == RS) slot_done = 0;
                }
            }
        }
#ifdef TNMF_TC_PROFILE
        prof_total += clock64();
        if (blockIdx.x == 0 && lane == 0)
            printf("hupd_ts mma X=%d: total %lld  wait x_free %lld  wait a_full %lld  wait turn %lld  issuing %lld\n", X, prof_total, prof_xfree, prof_afull, prof_turnw, prof_issue);
#endif
        __syncwarp();
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 8) tmem_dealloc(tmem_base, 512);
}

template <int KPT>
__global__ void __launch_bounds__(kThreads, 1) hupd_ts_kernel(const Geo2 g, const Plan p, const Args a) {
    hupd_ts_body<KPT, false>(g, p, a);
}
template <int KPT>
__global__ void __launch_bounds__(kThreads, 1) hupd_ts3_kernel(const Geo3 g, const Plan p, const Args a) {
    hupd_ts_body<KPT, true>(g, p, a);
}

template <int KPT> static auto kernel_for(const Geo2 &) { return hupd_ts_kernel<KPT>; }
template <int KPT> static auto kernel_for(const Geo3 &) { return hupd_ts3_kernel<KPT>; }

template <int KPT, class G>
static int launch(const G &g, const Plan &p, const Args &a, cudaStream_t st) {
    auto kern = kernel_for<KPT>(g);
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, kMaxSmem);
    if (e != cudaSuccess) return status_from_cuda(e);
    kern<<<(unsigned)p.grid, kThreads, p.smem, st>>>(g, p, a);
    TNMF_CHECK_LAUNCH();
    return TNMF_OK;
}

}  // namespace hut
}  // namespace tc

// ---- dispatch ----------------------------------------------------------------------------------------------------------
bool tc_hupd_ts_supported(const Geo &g, int dtype) {
    tc::hut::Plan p;
    if (plane_problem(g)) return tc::plane_mode_ok(g, dtype) && tc::hut::make_plan(tc::make_geo3(g, true), p);
    if (!tc::rank2_ok(g, dtype)) return false;
    return tc::hut::make_plan(tiled::make_geo2(g), p);
}

template <class G>
static int gradient_h_ts(const G &q, int M, const float *V, const float *R, const float *W, float *neg, float *pos,
                         float *H, double reg, const float *G_, double lambda, const float *Gsum, double lambda_cross,
                         cudaStream_t st) {
    tc::hut::Plan p;
    if (!tc::hut::make_plan(q, p)) return TNMF_EUNSUPPORTED;
    tc::hut::Args a;
    a.V = V; a.R = R; a.W = W; a.neg = neg; a.pos = pos; a.H = H;
    a.reg = (float)reg; a.lambda = (float)lambda; a.lambda_cross = (float)lambda_cross;
    a.G = G_; a.Gsum = Gsum;
    for (int m0 = 0; m0 < M; m0 += tc::hut::kNB) {
        a.m0 = m0;
        int s;
        switch (p.KP) {
            case 8: s = tc::hut::launch<8>(q, p, a, st); break;
            case 16: s = tc::hut::launch<16>(q, p, a, st); break;
            case 24: s = tc::hut::launch<24>(q, p, a, st); break;
            case 32: s = tc::hut::launch<32>(q, p, a, st); break;
            case 40: s = tc::hut::launch<40>(q, p, a, st); break;
            case 48: s = tc::hut::launch<48>(q, p, a, st); break;
            case 56: s = tc::hut::launch<56>(q, p, a, st); break;
            case 64: s = tc::hut::launch<64>(q, p, a, st); break;
            default: s = TNMF_EUNSUPPORTED;
        }
        if (s) return s;
    }
    return TNMF_OK;
}

int tc_gradient_h_ts(const Geo &g, const float *V, const float *R, const float *W, float *neg, float *pos, float *H,
                     double reg, const float *G, double lambda, const float *Gsum, double lambda_cross, cudaStream_t st,
                     int t_lo, int t_hi) {
    // 3-D: ONE launch per block of atoms - the a_z planes are channels of the contraction, so the fused epilogue sees
    // complete sums.  A plane window [t_lo, t_hi) makes the virtual samples (n, t_lo + t'), t' < t_hi - t_lo.
    if (plane_problem(g)) {
        tc::Geo3 q = tc::make_geo3(g, true);
        if (t_hi >= 0) {
            if (t_hi <= t_lo) return TNMF_OK;
            tc::window_geo3(q, g.N, t_lo, t_hi - t_lo);
        }
        return gradient_h_ts(q, g.M, V, R, W, neg, pos, H, reg, G, lambda, Gsum, lambda_cross, st);
    }
    if (t_hi >= 0) return TNMF_EUNSUPPORTED;
    return gradient_h_ts(tiled::make_geo2(g), g.M, V, R, W, neg, pos, H, reg, G, lambda, Gsum, lambda_cross, st);
}

int tc_hupd_ts_launches(const Geo &g) { return tiled::ceil_div(g.M, tc::hut::kNB); }

}  // namespace tnmf
