// Tensor-core (tcgen05, 3xTF32) H gradient with the fused multiplicative update.
//
//   neg[n,m,ty,tx] = sum_c sum_{ay,ax} W[m,c,ay,ax] * Vext[n,c,ty-offy+ay,tx-offx+ax]   (tnmf/backends/NumPy.py:101-109)
//   pos[n,m,ty,tx] = the same with R                                                    (tnmf/backends/NumPy.py:111-119)
//   epilogue (H given):  pos += lambda*(G-H); pos += lambda_c*(Gsum-G); pos += reg; H = (H*neg)/pos
//                                                           (tnmf/TransformInvariantNMF.py:217-235,246-271)
//
// Formulation.  A CTA owns a tile of 128 activation COLUMNS and walks down the rows.  Column J = n * TXP + xv lives
// in the flattened [N x TXP] space, TXP = TX + AX - 1: the AX-1 gap columns behind every sample (computed, never
// stored) make the source windows of different samples disjoint, so a tile may span samples and partial rows cost a
// few percent of the MMA lanes instead of a whole padded tile.  For a source
// row r of X (V or R) the "expander" warps build, once,
//       A_r[column i, k = (c, ax)] = Xext[n_i, c, r, tx_i - offx + ax]          128 x KP,  KP = roundup(C*AX, 8)
// in shared memory (canonical K-major no-swizzle layout, hi/lo TF32 split).  Source row r contributes to the output
// rows ty = r + offy - ay, ay = 0..AY-1, through
//       D_ty[column, m] += A_r[column, :] . Wt_ay[m, :]
// Output rows live in a ring of 16 TMEM slots (16 atoms x {neg, pos} = 32 columns each, 512 columns in all) and
// consecutive output rows occupy consecutive slots, so ONE tcgen05.mma with N = 16 * (number of live rows) serves all
// atom rows of the source row (the atom-row blocks of Wt are stored in that order).  3xTF32: hi*hi + lo*hi + hi*lo,
// FP32 accumulation in TMEM.  When the last source row of an output row has been issued, a tcgen05.commit hands the
// slot to the epilogue warps, which read it back (tcgen05.ld), apply the update and release the slot.
//
// Expansion: the source row segment of the tile (C x (128 + AX - 1) values, zero outside the sample) is fetched one
// stage ahead into registers, split into hi/lo once per element and parked in a small double-buffered "raw" array;
// every expander thread then copies its C*AX-wide window into the operand stage with LDS.32 / STS.128 only.
//
// Roles (448 threads): warps 0-7 expanders (thread = column x half of the K groups), warps 8-11 epilogue (thread =
// column = TMEM lane), warps 12 and 13 issue the MMAs of the V stages (neg accumulators) and of the R stages (pos) - converged warps, one
// elected lane issuing, because a single issuing thread cannot feed the tensor pipe at N <= 176.  mbarriers: a_full/a_empty per operand stage, row_done/slot_free per
// TMEM slot.  Atoms are processed in blocks of 16 (one launch per block).
// Bound: tensor pipe at the TF32 rate / 3 (DESIGN.md 3.4).
#include <cstdlib>
#include "tc_common.cuh"


namespace tnmf {
namespace tc {

using tiled::ceil_div;
using tiled::Geo2;
using tiled::round_up;

constexpr int kTile = 128;          // activation columns per CTA tile = MMA M
constexpr int kNB = 16;             // atoms per launch = MMA N granule
constexpr int kSlots = 16;          // TMEM ring: 16 output rows x (16 neg + 16 pos columns)
constexpr int kMaxStages = 6;
constexpr int kExpanders = 256;       // 8 expander warps: thread = (column, half of the K groups)
constexpr int kThreads = 32 * 14;     // 8 expander + 4 epilogue + 2 MMA-issuing warps
constexpr int kMaxSmem = 226 * 1024;
constexpr int kRawMax = 4;          // raw-row elements per expander thread (C * (128 + AX - 1) <= 1024)

struct TcHupdPlan {
    int KP, ksteps;                 // padded contraction length C*AX -> multiple of 8
    int TXP, RW, raw_floats, nraw;  // padded columns per sample, raw row width, floats per raw array, raw loads/thread
    int tiles, rblocks, rows_per_block;
    long long units;
    int n_stages, stage_floats, w_floats;
    int grid;
    size_t smem;
};

struct TcHupdArgs {
    const float *V, *R, *W;
    float *neg, *pos, *H;
    float reg, lambda, lambda_cross;
    const float *G, *Gsum;
    int m0;                         // first atom of this launch
};

bool make_tc_hupd_plan(const Geo2 &g, TcHupdPlan &p) {
    p = TcHupdPlan();
    if (g.AY > kSlots - 1 || g.AY < 1) return false;
    p.KP = round_up(g.C * g.AX, 8);
    if (p.KP > 64) return false;                            // KGT <= 16
    p.ksteps = p.KP / 8;
    p.stage_floats = 2 * kTile * p.KP;                     // hi + lo
    p.w_floats = 2 * g.AY * kNB * p.KP;                    // hi + lo, atom-row blocks in ring order
    p.TXP = g.TX + g.AX - 1;
    p.RW = kTile + g.AX - 1;
    p.raw_floats = round_up(g.C * p.RW + kTile, 32);        // + 128 zeros read by the padded k
    p.nraw = ceil_div(g.C * p.RW, kExpanders);
    if (p.nraw > kRawMax) return false;
    const size_t fixed = (size_t)p.w_floats * 4 + (size_t)4 * p.raw_floats * 4 + 1024;
    if (fixed + 2 * (size_t)p.stage_floats * 4 > (size_t)kMaxSmem) return false;
    p.n_stages = (int)(((size_t)kMaxSmem - fixed) / ((size_t)p.stage_floats * 4));
    if (p.n_stages > kMaxStages) p.n_stages = kMaxStages;
    p.n_stages &= ~1;                                       // V stages even, R stages odd: one issuing warp each
    p.smem = fixed + (size_t)p.n_stages * p.stage_floats * 4;
    const long long cols = (long long)g.N * p.TXP;
    if (cols <= 0 || cols >= (1ll << 31) - kTile) return false;
    p.tiles = (int)((cols + kTile - 1) / kTile);
    // row blocks: minimise waves * (rows + per-unit overhead)
    const int sms = tma::sm_count();
    double best = -1;
    for (int rb = 1; rb <= g.TY && rb <= 64; ++rb) {
        const int rows = ceil_div(g.TY, rb);
        if (ceil_div(g.TY, rows) != rb) continue;
        const long long units = (long long)p.tiles * rb;
        const double waves = (double)((units + sms - 1) / sms);
        const double cost = waves * (rows + 0.3 * (g.AY - 1) + 1.0);
        if (best < 0 || cost < best * 0.999) { best = cost; p.rblocks = rb; p.rows_per_block = rows; }
    }
    p.units = (long long)p.tiles * p.rblocks;
    p.grid = (int)(p.units < sms ? p.units : sms);
    return true;
}

struct Unit {
    int tile, ty0, ty1, r_lo, r_hi;
};
__device__ __forceinline__ Unit make_unit(long long u, const Geo2 &g, const TcHupdPlan &p) {
    Unit w;
    const int rb = (int)(u / p.tiles);
    w.tile = (int)(u - (long long)rb * p.tiles);
    w.ty0 = rb * p.rows_per_block;
    w.ty1 = min(g.TY, w.ty0 + p.rows_per_block);
    w.r_lo = max(0, w.ty0 - g.offy);
    w.r_hi = min(g.DY - 1, w.ty1 - 1 - g.offy + g.AY - 1);
    return w;
}

// KGH: compile-time bound on the 16-byte K groups one expander thread copies (ceil(KP / 8) <= KGH)
template <int KGH>
__global__ void __launch_bounds__(kThreads, 1)
hupd_tc_kernel(const Geo2 g, const TcHupdPlan p, const TcHupdArgs a) {
    extern __shared__ __align__(128) float smem[];
    __shared__ __align__(8) unsigned long long a_full[kMaxStages], a_empty[kMaxStages], row_done[kSlots],
        slot_free[kSlots];
    __shared__ unsigned tmem_base_s;
    // warp index out of a shuffle: ptxas then knows the role branches are warp-uniform and keeps the MMA issuers' operands in
    // uniform registers (tc_gradw_ts.cu has the measurements)
    const int tid = threadIdx.x, warp = __shfl_sync(0xffffffffu, tid >> 5, 0), lane = tid & 31;
    const int KP = p.KP, AY = g.AY, AX = g.AX, C = g.C;
    const int NR = AY * kNB;                               // rows of the atom operand
    float *w_hi = smem, *w_lo = smem + NR * KP;
    float *raw = smem + p.w_floats;                         // [2 buffers][hi, lo][raw_floats]
    float *stages = raw + 4 * p.raw_floats;
    __shared__ __align__(16) int koff[64];                                // k -> offset of (c, ax) in a raw array (padding -> zeros)
    const int RW = p.RW;
    if (tid < KP) koff[tid] = tid < C * AX ? (tid / AX) * RW + (tid % AX) : C * RW;
    for (int idx = tid; idx < 4 * kTile; idx += kThreads) raw[(idx / kTile) * p.raw_floats + C * RW + (idx % kTile)] = 0.f;

    if (tid == 0) {
        for (int s = 0; s < p.n_stages; ++s) { mbar_init(&a_full[s], kExpanders); mbar_init(&a_empty[s], 1); }
        for (int s = 0; s < kSlots; ++s) { mbar_init(&row_done[s], 2); mbar_init(&slot_free[s], kTile); }
        mbar_fence_init();
    }
    if (warp == 12) tmem_alloc(&tmem_base_s, 512);
    // atom operand: row n = j*16 + ml  <->  atom m0+ml, atom row ay = AY-1-j;  k = c*AX + ax
    for (int idx = tid; idx < NR * KP; idx += kThreads) {
        const int n = idx / KP, k = idx - n * KP;
        const int j = n / kNB, ml = n - j * kNB;
        const int m = a.m0 + ml, ay = AY - 1 - j;
        float v = 0.f;
        if (m < g.M && k < C * AX) {
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

    if (warp < 8) {
        // ------------------------------------ expanders ------------------------------------
        const int i = tid & (kTile - 1), half = tid >> 7;
        int st = 0;
        unsigned ph = 0, buf = 0;
        TC_PROF_DECL(empty); TC_PROF_DECL(bar); TC_PROF_DECL(total);
#ifdef TNMF_TC_PROFILE
        prof_total = -clock64();
#endif
        const long long plane = (long long)g.DY * g.DX;
        const int KG = KP >> 2;
        const int kg0 = half * ((KG + 1) >> 1), kg1 = half ? KG : ((KG + 1) >> 1);   // this thread's K groups
        const int raw_count = C * RW;
        int4 ko[KGH];                           // raw-array offsets of the 4 k of every K group (same for all stages)
#pragma unroll
        for (int j = 0; j < KGH; ++j)
            ko[j] = kg0 + j < kg1 ? *reinterpret_cast<const int4 *>(&koff[4 * (kg0 + j)]) : make_int4(0, 0, 0, 0);
        for (long long u = blockIdx.x; u < p.units; u += gridDim.x) {
            const Unit w = make_unit(u, g, p);
            // source element of every raw slot (q = tid + 256 e -> channel q / RW, position q % RW) in row 0, or -1: zero
            long long roff[kRawMax];
#pragma unroll
            for (int e = 0; e < kRawMax; ++e) {
                roff[e] = -1;
                const int q = tid + kExpanders * e;
                if (e < p.nraw && q < raw_count) {
                    const int c = q / RW;
                    const long long J = (long long)w.tile * kTile + (q - c * RW);
                    const int n = (int)(J / p.TXP);
                    const int x = (int)(J - (long long)n * p.TXP) - g.offx;
                    if (n < g.N && (unsigned)x < (unsigned)g.DX) roff[e] = ((long long)n * C + c) * plane + x;
                }
            }
            float rv[kRawMax];
            auto load_raw = [&](int sidx) {
                const float *src = ((sidx & 1) ? a.R : a.V) + (long long)(w.r_lo + (sidx >> 1)) * g.DX;
#pragma unroll
                for (int e = 0; e < kRawMax; ++e) rv[e] = roff[e] >= 0 ? __ldg(src + roff[e]) : 0.f;
            };
            const int n_st = 2 * (w.r_hi - w.r_lo + 1);
            load_raw(0);
            for (int sidx = 0; sidx < n_st; ++sidx) {
                float *raw_hi = raw + (size_t)buf * 2 * p.raw_floats, *raw_lo = raw_hi + p.raw_floats;
#pragma unroll
                for (int e = 0; e < kRawMax; ++e) {
                    if (e < p.nraw && tid + kExpanders * e < raw_count) {
                        float hi, lo;
                        split_tf32(rv[e], hi, lo);
                        raw_hi[tid + kExpanders * e] = hi;
                        raw_lo[tid + kExpanders * e] = lo;
                    }
                }
                if (sidx + 1 < n_st) load_raw(sidx + 1);             // in flight while this stage is expanded
                TC_PROF_WAIT(bar, asm volatile("bar.sync 1, 256;\n" ::: "memory"));
                TC_PROF_WAIT(empty, mbar_wait_backoff(&a_empty[st], ph ^ 1u, 40));
                float *d_hi = stages + (size_t)st * p.stage_floats + (size_t)(i >> 3) * 32 + (size_t)(i & 7) * 4 +
                              (size_t)kg0 * (kTile * 4);
                float *d_lo = d_hi + kTile * KP;
                const float *s_hi = raw_hi + i, *s_lo = raw_lo + i;
                // two K groups per batch: 16 independent LDS in flight before the 4 STS.128
#pragma unroll
                for (int j = 0; j < KGH; j += 2) {
                    if (kg0 + j < kg1) {
                        const int4 o0 = ko[j];
                        const float4 h0 = make_float4(s_hi[o0.x], s_hi[o0.y], s_hi[o0.z], s_hi[o0.w]);
                        const float4 l0 = make_float4(s_lo[o0.x], s_lo[o0.y], s_lo[o0.z], s_lo[o0.w]);
                        if (j + 1 < KGH && kg0 + j + 1 < kg1) {
                            const int4 o1 = ko[j + 1 < KGH ? j + 1 : j];
                            const float4 h1 = make_float4(s_hi[o1.x], s_hi[o1.y], s_hi[o1.z], s_hi[o1.w]);
                            const float4 l1 = make_float4(s_lo[o1.x], s_lo[o1.y], s_lo[o1.z], s_lo[o1.w]);
                            *reinterpret_cast<float4 *>(d_hi + (size_t)(j + 1) * (kTile * 4)) = h1;
                            *reinterpret_cast<float4 *>(d_lo + (size_t)(j + 1) * (kTile * 4)) = l1;
                        }
                        *reinterpret_cast<float4 *>(d_hi + (size_t)j * (kTile * 4)) = h0;
                        *reinterpret_cast<float4 *>(d_lo + (size_t)j * (kTile * 4)) = l0;
                    }
                }
                fence_proxy_async();
                mbar_arrive(&a_full[st]);
                if (++st == p.n_stages) { st = 0; ph ^= 1u; }
                buf ^= 1u;
            }
        }
#ifdef TNMF_TC_PROFILE
        prof_total += clock64();
        if (blockIdx.x == 0 && tid == 0)
            printf("expander: total %lld  wait a_empty %lld  raw barrier %lld\n", prof_total, prof_empty, prof_bar);
#endif
    } else if (warp < 12) {
        // ------------------------------------ epilogue ------------------------------------
        const int i = tid - kExpanders;
        const unsigned lane_base = (unsigned)((warp & 3) * 32) << 16;
        const long long tvol = (long long)g.TY * g.TX;
        long long g_base = 0;
        TC_PROF_DECL(done); TC_PROF_DECL(total); TC_PROF_DECL(ldtm); TC_PROF_DECL(arrive);
#ifdef TNMF_TC_PROFILE
        prof_total = -clock64();
#endif
        for (long long u = blockIdx.x; u < p.units; u += gridDim.x) {
            const Unit w = make_unit(u, g, p);
            const long long J = (long long)w.tile * kTile + i;
            const int n = (int)(J / p.TXP);
            const int tx = (int)(J - (long long)n * p.TXP);
            const bool active = n < g.N && tx < g.TX;
            // the activations of a row do not depend on the accumulators: they are fetched one row ahead
            float hnext[kNB];
            float *hrow = (a.H && active) ? a.H + (long long)n * g.hsn + (long long)a.m0 * g.hsm + tx : nullptr;
            auto load_h = [&](int ty) {
#pragma unroll
                for (int ml = 0; ml < kNB; ++ml)
                    hnext[ml] = (hrow && a.m0 + ml < g.M) ? hrow[(long long)ty * g.hsy + (long long)ml * g.hsm] : 0.f;
            };
            const bool fast = a.H && !a.G && a.m0 + kNB <= g.M;
            load_h(w.ty0);
            for (int ty = w.ty0; ty < w.ty1; ++ty) {
                const long long gi = g_base + (ty - w.ty0);
                const int s = (int)(gi & (kSlots - 1));
                const unsigned par = (unsigned)((gi >> 4) & 1);
                TC_PROF_WAIT(done, mbar_wait_backoff(&row_done[s], par, 100));
                tc_fence_after();
                float neg[kNB], pos[kNB];
                TC_PROF_WAIT(ldtm, tmem_ld16(tmem_base + lane_base + (unsigned)(s * kNB), neg);
                             tmem_ld16(tmem_base + lane_base + 256u + (unsigned)(s * kNB), pos); tmem_ld_wait());
                tc_fence_before();
                TC_PROF_WAIT(arrive, mbar_arrive(&slot_free[s]));
                float hv[kNB];
#pragma unroll
                for (int ml = 0; ml < kNB; ++ml) hv[ml] = hnext[ml];
                if (fast) {
                    // plain fused update of a full block of 16 atoms: pointer walks, no per-atom tests.  The product and the
                    // quotient round separately and to nearest, like the reference's `arr *= neg; arr /= pos`.
                    if (active) {
                        float *o = hrow + (long long)ty * g.hsy;
                        if (ty + 1 < w.ty1) {
                            const float *q = o + g.hsy;
#pragma unroll
                            for (int ml = 0; ml < kNB; ++ml) { hnext[ml] = *q; q += g.hsm; }
                        }
#pragma unroll
                        for (int ml = 0; ml < kNB; ++ml) {
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
                for (int ml = 0; ml < kNB; ++ml) {
                    const int m = a.m0 + ml;
                    if (m >= g.M) continue;
                    const long long cidx = ((long long)n * g.M + m) * tvol + tin;
                    if (a.H) {
                        const float h = hv[ml];
                        float ps = pos[ml];
                        if (a.G) {
                            const float gv = a.G[cidx];
                            if (a.lambda != 0.f) { float tmp = gv - h; tmp *= a.lambda; ps += tmp; }
                            if (a.Gsum) {
                                const float gs = a.Gsum[(long long)n * tvol + tin];
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
            g_base += w.ty1 - w.ty0;
        }
#ifdef TNMF_TC_PROFILE
        prof_total += clock64();
        if (blockIdx.x == 0 && i == 0) printf("epilogue: total %lld  wait row_done %lld  ldtm %lld  arrive %lld\n", prof_total, prof_done, prof_ldtm, prof_arrive);
#endif
    } else {
      {
        // ------------------------------------ MMA issuer ------------------------------------
        // the whole warp walks the schedule (converged, uniform registers); one elected lane issues
        // descriptors: only the 14-bit start-address field changes between MMAs, so they are kept as (lo, hi) words
        const unsigned lbo_a = kTile * 16, lbo_b = (unsigned)NR * 16;
        const unsigned desc_hi = (128u >> 4) | (1u << 14);                      // SBO, descriptor version 1
        const unsigned a_lo_word = ((lbo_a >> 4) << 16), b_lo_word = ((lbo_b >> 4) << 16);
        const unsigned w_hi16 = __shfl_sync(0xffffffffu, smem_u32(w_hi) >> 4, 0), w_lo16 = __shfl_sync(0xffffffffu, smem_u32(w_lo) >> 4, 0);
        const unsigned w_addr16[3] = {w_hi16, w_hi16, w_lo16};
        const unsigned stage_addr0 = __shfl_sync(0xffffffffu, smem_u32(stages), 0);
        const unsigned tmem_u = __shfl_sync(0xffffffffu, tmem_base, 0);
        const unsigned a_step16 = (2 * lbo_a) >> 4, b_step16 = (2 * lbo_b) >> 4;
        const int x = warp - 12;                // warp 12 issues the V stages (neg accumulators), warp 13 the R stages (pos)
        int st = x;
        unsigned ph = 0;
        long long g_base = 0;
        TC_PROF_DECL(full); TC_PROF_DECL(slot); TC_PROF_DECL(total);
#ifdef TNMF_TC_PROFILE
        prof_total = -clock64();
#endif
        for (long long u = blockIdx.x; u < p.units; u += gridDim.x) {
            const Unit w = make_unit(u, g, p);
            int next_new = w.ty0, next_done = w.ty0;
            for (int r = w.r_lo; r <= w.r_hi; ++r) {
                const int ay_lo = max(0, r + g.offy - (w.ty1 - 1)), ay_hi = min(AY - 1, r + g.offy - w.ty0);
                const int t_a = r + g.offy - ay_hi, t_b = r + g.offy - ay_lo;
                const int j0 = r + g.offy - AY + 1;                 // output row of atom-row block 0
                // output rows that receive their first contribution from this source row: [first_new, t_b]
                const int first_new = next_new;
                for (; next_new <= t_b; ++next_new) {
                    const long long gi = g_base + (next_new - w.ty0);
                    if (gi >= kSlots)
                        TC_PROF_WAIT(slot, mbar_wait(&slot_free[gi & (kSlots - 1)], (unsigned)(((gi >> 4) - 1) & 1)));
                }
                tc_fence_after();
                // the MMAs of this source row: up to two column runs of the ring for the rows that accumulate ...
                unsigned o_col[2], o_idesc[2], o_b16[2];
                int n_ops = 0;
                auto add_ops = [&](int lo, int hi, unsigned *col, unsigned *idesc, unsigned *b16, int &n) {
                    if (lo > hi) return;
                    const int cnt = hi - lo + 1;
                    const int s = (int)((g_base + (lo - w.ty0)) & (kSlots - 1));
                    const int first = min(cnt, kSlots - s);
                    col[n] = (unsigned)(s * kNB); idesc[n] = idesc_tf32(kTile, kNB * first);
                    b16[n] = (unsigned)(lo - j0) * 16u; ++n;
                    if (cnt > first) {
                        col[n] = 0u; idesc[n] = idesc_tf32(kTile, kNB * (cnt - first));
                        b16[n] = (unsigned)(lo - j0 + first) * 16u; ++n;
                    }
                };
                add_ops(t_a, t_b, o_col, o_idesc, o_b16, n_ops);
                // ... and, for the very first MMA of the row, the same split into old rows (accumulate) / new rows (overwrite)
                unsigned f_col[4], f_idesc[4], f_b16[4];
                int n_old = 0, n_first = 0;
                if (first_new <= t_b) {
                    add_ops(t_a, first_new - 1, f_col, f_idesc, f_b16, n_first);
                    n_old = n_first;
                    add_ops(max(first_new, t_a), t_b, f_col, f_idesc, f_b16, n_first);
                }
                {
                    TC_PROF_WAIT(full, mbar_wait(&a_full[st], ph));
                    tc_fence_after();
                    const unsigned col_base = tmem_u + (x ? 256u : 0u);
                    const unsigned a_hi16 = (stage_addr0 + (unsigned)st * (unsigned)p.stage_floats * 4u) >> 4;
                    const unsigned a_addr16[3] = {a_hi16, a_hi16 + ((kTile * KP * 4u) >> 4), a_hi16};
                    if (elect_one()) {              // one election per stage: operands go to uniform registers once
                        for (int ks = 0; ks < p.ksteps; ++ks) {
#pragma unroll
                            for (int t = 0; t < 3; ++t) {
                                const unsigned long long da =
                                    ((unsigned long long)desc_hi << 32) | (a_lo_word | (a_addr16[t] + ks * a_step16));
                                const unsigned b16 = w_addr16[t] + ks * b_step16;
                                if (ks == 0 && t == 0 && n_first > 0) {
#pragma unroll
                                    for (int o = 0; o < 4; ++o)
                                        if (o < n_first)
                                            mma_tf32(col_base + f_col[o], da,
                                                     ((unsigned long long)desc_hi << 32) | (b_lo_word | (b16 + f_b16[o])),
                                                     f_idesc[o], o < n_old ? 1u : 0u);
                                } else {
                                    mma_tf32(col_base + o_col[0], da,
                                             ((unsigned long long)desc_hi << 32) | (b_lo_word | (b16 + o_b16[0])), o_idesc[0], 1u);
                                    if (n_ops > 1)
                                        mma_tf32(col_base + o_col[1], da,
                                                 ((unsigned long long)desc_hi << 32) | (b_lo_word | (b16 + o_b16[1])),
                                                 o_idesc[1], 1u);
                                }
                            }
                        }
                    }
                    __syncwarp();
                    mma_commit_elect(&a_empty[st]);
                    st += 2;
                    if (st >= p.n_stages) { st = x; ph ^= 1u; }
                }
                // output rows whose last source row this was (the barrier needs the commit of both issuing warps)
                for (; next_done < w.ty1 && min(g.DY - 1, next_done - g.offy + AY - 1) <= r; ++next_done)
                    mma_commit_elect(&row_done[(g_base + (next_done - w.ty0)) & (kSlots - 1)]);
            }
            g_base += w.ty1 - w.ty0;
        }
#ifdef TNMF_TC_PROFILE
        prof_total += clock64();
        if (blockIdx.x == 0 && lane == 0 && x == 0)
            printf("mma: total %lld  wait a_full %lld  wait slot_free %lld\n", prof_total, prof_full, prof_slot);
#endif
      }
      __syncwarp();
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 12) tmem_dealloc(tmem_base, 512);
}

template <int KGH>
static int launch(const Geo2 &g, const TcHupdPlan &p, const TcHupdArgs &a, cudaStream_t st) {
    auto kern = hupd_tc_kernel<KGH>;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, kMaxSmem);
    if (e != cudaSuccess) return status_from_cuda(e);
    kern<<<(unsigned)p.grid, kThreads, p.smem, st>>>(g, p, a);
    TNMF_CHECK_LAUNCH();
    return TNMF_OK;
}

}  // namespace tc

// ---- dispatch ----------------------------------------------------------------------------------------------------------
bool tc_hupd_supported(const Geo &g, int dtype) {
    if (!tc::rank2_ok(g, dtype)) return false;
    tc::TcHupdPlan p;
    return tc::make_tc_hupd_plan(tiled::make_geo2(g), p);
}

int tc_gradient_h(const Geo &g, const float *V, const float *R, const float *W, float *neg, float *pos, float *H,
                  double reg, const float *G, double lambda, const float *Gsum, double lambda_cross, cudaStream_t st) {
    const tiled::Geo2 q = tiled::make_geo2(g);
    tc::TcHupdPlan p;
    if (!tc::make_tc_hupd_plan(q, p)) return TNMF_EUNSUPPORTED;
    tc::TcHupdArgs a;
    a.V = V; a.R = R; a.W = W; a.neg = neg; a.pos = pos; a.H = H;
    a.reg = (float)reg; a.lambda = (float)lambda; a.lambda_cross = (float)lambda_cross;
    a.G = G; a.Gsum = Gsum;
    for (int m0 = 0; m0 < g.M; m0 += tc::kNB) {
        a.m0 = m0;
        int s;
        const int kgh = (p.KP / 4 + 1) / 2;                 // K groups per expander thread
        if (kgh <= 1) s = tc::launch<1>(q, p, a, st);
        else if (kgh <= 2) s = tc::launch<2>(q, p, a, st);
        else if (kgh <= 3) s = tc::launch<3>(q, p, a, st);
        else if (kgh <= 4) s = tc::launch<4>(q, p, a, st);
        else if (kgh <= 5) s = tc::launch<5>(q, p, a, st);
        else if (kgh <= 6) s = tc::launch<6>(q, p, a, st);
        else if (kgh <= 8) s = tc::launch<8>(q, p, a, st);
        else s = TNMF_EUNSUPPORTED;
        if (s) return s;
    }
    return TNMF_OK;
}

int tc_hupd_launches(const Geo &g) { return tiled::ceil_div(g.M, tc::kNB); }

}  // namespace tnmf
