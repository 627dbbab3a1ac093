// tcgen05 / TMEM primitives for the tensor-core kernels (sm_100a), hand-written PTX.
//
// Operand layout used throughout: the canonical K-major, no-swizzle ("interleaved") shared-memory layout of the
// tcgen05 matrix descriptors for 32-bit elements.  A matrix of `rows` x K floats is stored as 8-row x 16-byte core
// matrices; element (i, k) lives at byte offset
//       (i / 8) * 128  +  (k / 4) * (rows * 16)  +  (i % 8) * 16  +  (k % 4) * 4
// i.e. stride-byte-offset (between 8-row groups) = 128 and leading-byte-offset (between the 16-byte K chunks) =
// rows * 16.  One kind::tf32 MMA consumes K = 8 (two 16-byte chunks); consecutive K steps advance the descriptor's
// start address by 2 * LBO.  A row group offset advances it by 128 bytes per 8 rows.
#pragma once
#include <cstdint>
#include "tma_common.cuh"

// -DTNMF_TC_PROFILE: CTA 0 prints, per role, the cycles it spent blocked on each of its barriers (debug builds only)
#ifdef TNMF_TC_PROFILE
#include <cstdio>
#define TC_PROF_DECL(n) long long prof_##n = 0
#define TC_PROF_WAIT(n, stmt) do { const long long t__ = clock64(); stmt; prof_##n += clock64() - t__; } while (0)
#else
#define TC_PROF_DECL(n)
#define TC_PROF_WAIT(n, stmt) stmt
#endif

namespace tnmf {
namespace tc {

using tma::mbar_arrive;
using tma::mbar_fence_init;
using tma::mbar_init;
using tma::mbar_wait;
using tma::smem_u32;

// ---- plane mode: 3-D 'valid' problems on the 2-D tensor-memory kernels (DESIGN.md §3.10) ----------------------------
// In 'valid' mode a 3-D correlation is a sum over the atom plane a_z of 2-D correlations between z-planes, so the 2-D
// kernels run over VIRTUAL SAMPLES nv = n * NZ + z (one z-plane of sample n each) with a two-level address:
//   V / R plane z of sample n, channel c:  n * xsn + c * xsc + z * D_y * D_x
//   H plane t of sample n, atom m:         n * hsn + m * hsm + t * hsz
// The reconstruction and the W gradient launch once per a_z (NZ = D_z, H shifted by offz - az planes); the H update
// launches once, its a_z planes being extra channels (c, a_z) of the contraction (NZ = T_z, Geo2::C = C * A_z).
// A plane window (tnmf_update_h_planes / tnmf_gradient_w_planes) runs over the virtual samples (n, z0 + z'), z' < NZ: the
// H update over the activation planes [z0, z0 + NZ) = [t_lo, t_hi), each W-gradient launch over the sample planes whose
// activation plane lies in the window.  Every address and boundary test uses the absolute plane z0 + z'.
struct Geo3 : tiled::Geo2 {
    int NZ;                 // planes per sample in the virtual sample index
    int z0;                 // absolute plane of z' = 0 (0 without a window)
    int TZ;                 // activation planes of the whole problem (the pitch of the dense G / Gsum inputs)
    int DZ, AZ, offz;       // sample planes, atom planes, A_z - 1
    int az;                 // atom plane of this launch (reconstruction, W gradient)
    int acc;                // reconstruction: add to R instead of writing it (every launch after the first)
    long long xsn, xsc;     // element strides of V / R between samples and between channels
    long long hsz;          // element stride between activation planes (T_y * hsy)
};

// 2-D problems the tensor-core kernels serve: float32, not 'circular', rank <= 2 but not rank 1 (the FP32 kernels serve
// that), at least one sample
inline bool rank2_ok(const Geo &g, int dtype) {
    if (dtype != TNMF_F32 || g.wrap || g.N < 1) return false;
    return g.D[0] == 1 && g.A[0] == 1 && g.T[0] == 1 && !(g.D[1] == 1 && g.A[1] == 1);
}
// 3-D problems the plane mode serves: float32 'valid' (off = A - 1 on every axis)
inline bool plane_mode_ok(const Geo &g, int dtype) {
    if (dtype != TNMF_F32 || g.wrap || !plane_problem(g) || g.N < 1) return false;
    for (int i = 0; i < 3; ++i)
        if (g.off[i] != g.A[i] - 1 || g.T[i] != g.D[i] + g.A[i] - 1) return false;
    return true;
}
// h_update: virtual samples over the activation planes, virtual channels (c, a_z); otherwise over the sample planes
inline Geo3 make_geo3(const Geo &g, bool h_update, int az = 0) {
    Geo3 q;
    static_cast<tiled::Geo2 &>(q) = tiled::make_geo2(g);
    q.NZ = h_update ? g.T[0] : g.D[0];
    q.N = g.N * q.NZ;
    q.z0 = 0;
    q.TZ = g.T[0];
    if (h_update) q.C = g.C * g.A[0];
    q.DZ = g.D[0]; q.AZ = g.A[0]; q.offz = g.off[0];
    q.az = az; q.acc = 0;
    q.xsc = (long long)g.D[0] * g.D[1] * g.D[2];
    q.xsn = q.xsc * g.C;
    q.hsz = (long long)g.T[1] * g.hsy;
    return q;
}
// the same geometry restricted to the planes [z0, z0 + nz) of the virtual sample index
inline void window_geo3(Geo3 &q, int n_samples, int z0, int nz) {
    q.z0 = z0;
    q.NZ = nz;
    q.N = n_samples * nz;
}

// Wait with back-off for roles that are far from the critical path: every poll of a spinning warp is a shared-memory
// wavefront, and shared-memory bandwidth is what bounds the tensor-core kernels (ncu: polls were 30% of the LSU traffic).
__device__ __forceinline__ void mbar_wait_backoff(unsigned long long *bar, unsigned parity, unsigned ns) {
    while (!tma::mbar_try_wait(bar, parity)) __nanosleep(ns);
}

__device__ __forceinline__ size_t canon_offset_floats(int i, int k, int rows) {
    return (size_t)(i >> 3) * 32 + (size_t)(k >> 2) * ((size_t)rows * 4) + (size_t)(i & 7) * 4 + (size_t)(k & 3);
}

// 64-bit shared-memory matrix descriptor: start address, LBO, SBO (all >> 4), descriptor version 1 (Blackwell),
// base offset 0, layout type 0 (no swizzle).
__device__ __forceinline__ unsigned long long smem_desc(unsigned addr_bytes, unsigned lbo_bytes, unsigned sbo_bytes) {
    unsigned long long d = 0;
    d |= (unsigned long long)((addr_bytes >> 4) & 0x3FFFu);
    d |= (unsigned long long)((lbo_bytes >> 4) & 0x3FFFu) << 16;
    d |= (unsigned long long)((sbo_bytes >> 4) & 0x3FFFu) << 32;
    d |= 1ull << 46;
    return d;
}

// 32-bit instruction descriptor of kind::tf32: D = F32, A = B = TF32, both K-major, dense, M x N.
__host__ __device__ constexpr unsigned idesc_tf32(int m, int n) {
    return (1u << 4) | (2u << 7) | (2u << 10) | ((unsigned)(n >> 3) << 17) | ((unsigned)(m >> 4) << 24);
}

// D[tmem] (+)= A[smem] * B[smem]^T, issued by ONE thread.
__device__ __forceinline__ void mma_tf32(unsigned tmem_d, unsigned long long desc_a, unsigned long long desc_b,
                                         unsigned idesc, unsigned accumulate) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n"
        "}\n" ::"r"(tmem_d),
        "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
}

// The same, executed by a whole converged warp: one elected lane issues.  Keeping the issuing warp converged lets the
// compiler hold descriptors and addresses in uniform registers (a divergent `if (lane == 0)` costs an R2UR +
// election loop around every MMA: measured 175 clk per MMA against 46 for the bare instruction).
__device__ __forceinline__ void mma_tf32_elect(unsigned tmem_d, unsigned long long desc_a, unsigned long long desc_b,
                                               unsigned idesc, unsigned accumulate) {
    asm volatile(
        "{\n"
        ".reg .pred p, q;\n"
        "elect.sync _|q, 0xffffffff;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "@q tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n"
        "}\n" ::"r"(tmem_d),
        "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
}
// The same with the A operand in TENSOR MEMORY (lane = operand row, 32-bit column = one K element; the column address must
// be a multiple of 4).  Measured on B200 (tools/tc_probe2.cu): 128 x N x 8 takes N/2 clk from N = 48 on - no operand-fetch
// floor (the shared-memory form needs >= 44 clk for its 4 KB A operand) and no A traffic on the shared-memory port.
__device__ __forceinline__ void mma_tf32_ts_elect(unsigned tmem_d, unsigned tmem_a, unsigned long long desc_b, unsigned idesc,
                                                  unsigned accumulate) {
    asm volatile(
        "{\n"
        ".reg .pred p, q;\n"
        "elect.sync _|q, 0xffffffff;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "@q tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n"
        "}\n" ::"r"(tmem_d),
        "r"(tmem_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
}
// One lane of a converged warp (for `if (elect_one()) { several MMAs }`: the operands are moved to uniform registers once
// per branch instead of once per instruction, as the per-instruction election of mma_tf32*_elect forces)
__device__ __forceinline__ bool elect_one() {
    unsigned pred;
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "elect.sync _|p, 0xffffffff;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n"
        : "=r"(pred));
    return pred != 0;
}
__device__ __forceinline__ void mma_tf32_ts(unsigned tmem_d, unsigned tmem_a, unsigned long long desc_b, unsigned idesc,
                                            unsigned accumulate) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n"
        "}\n" ::"r"(tmem_d),
        "r"(tmem_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
}
// Same, the B descriptor given as its two 32-bit words (only the low word - start address | LBO - changes between MMAs, so
// the issuing loop advances it with one uniform add) and always accumulating / never accumulating.
template <bool kAccumulate>
__device__ __forceinline__ void mma_tf32_ts2(unsigned tmem_d, unsigned tmem_a, unsigned desc_b_lo, unsigned desc_b_hi,
                                             unsigned idesc) {
    if constexpr (kAccumulate)
        asm volatile(
            "{\n"
            ".reg .b64 d;\n"
            ".reg .pred p;\n"
            "mov.b64 d, {%2, %3};\n"
            "setp.eq.b32 p, 0, 0;\n"
            "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], d, %4, p;\n"
            "}\n" ::"r"(tmem_d),
            "r"(tmem_a), "r"(desc_b_lo), "r"(desc_b_hi), "r"(idesc)
            : "memory");
    else
        asm volatile(
            "{\n"
            ".reg .b64 d;\n"
            ".reg .pred p;\n"
            "mov.b64 d, {%2, %3};\n"
            "setp.ne.b32 p, 0, 0;\n"
            "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], d, %4, p;\n"
            "}\n" ::"r"(tmem_d),
            "r"(tmem_a), "r"(desc_b_lo), "r"(desc_b_hi), "r"(idesc)
            : "memory");
}
__device__ __forceinline__ void mma_commit_elect(unsigned long long *bar) {
    asm volatile(
        "{\n"
        ".reg .pred q;\n"
        "elect.sync _|q, 0xffffffff;\n"
        "@q tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n"
        "}\n" ::"r"(smem_u32(bar))
        : "memory");
}

// mbarrier arrive once all tcgen05 operations issued so far by this thread have completed (implies
// tcgen05.fence::before_thread_sync).
__device__ __forceinline__ void mma_commit(unsigned long long *bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n" ::"r"(smem_u32(bar))
                 : "memory");
}

__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory"); }
// generic-proxy shared-memory writes -> visible to the async proxy (the tensor core reads operands through it)
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory"); }

// Whole-warp TMEM allocation of `cols` columns (power of two >= 32); the base address lands in *slot (shared).
__device__ __forceinline__ void tmem_alloc(unsigned *slot, unsigned cols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;\n" ::"r"(smem_u32(slot)), "r"(cols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;\n" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(unsigned base, unsigned cols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;\n" ::"r"(base), "r"(cols) : "memory");
}

// 16 consecutive columns of this thread's TMEM lane (lane = 32 * (warp % 4) + laneid) -> 16 registers.
__device__ __forceinline__ void tmem_ld16(unsigned addr, float (&v)[16]) {
    unsigned r[16];
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, "
        "[%16];\n"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(addr)
        : "memory");
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}
__device__ __forceinline__ void tmem_ld8(unsigned addr, float (&v)[8]) {
    unsigned r[8];
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];\n"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
                 : "r"(addr)
                 : "memory");
#pragma unroll
    for (int i = 0; i < 8; ++i) v[i] = __uint_as_float(r[i]);
}
__device__ __forceinline__ void tmem_st8_zero(unsigned addr) {
    const unsigned z = 0u;
    asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %1, %1, %1, %1, %1, %1, %1};\n" ::"r"(addr), "r"(z) : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;\n" ::: "memory"); }

// 16 / 8 registers -> consecutive columns of this thread's TMEM lane (whole warp, lanes 32 * (warp % 4) + laneid)
__device__ __forceinline__ void tmem_st16(unsigned addr, const float (&v)[16]) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};\n" ::
            "r"(addr),
        "r"(__float_as_uint(v[0])), "r"(__float_as_uint(v[1])), "r"(__float_as_uint(v[2])), "r"(__float_as_uint(v[3])),
        "r"(__float_as_uint(v[4])), "r"(__float_as_uint(v[5])), "r"(__float_as_uint(v[6])), "r"(__float_as_uint(v[7])),
        "r"(__float_as_uint(v[8])), "r"(__float_as_uint(v[9])), "r"(__float_as_uint(v[10])), "r"(__float_as_uint(v[11])),
        "r"(__float_as_uint(v[12])), "r"(__float_as_uint(v[13])), "r"(__float_as_uint(v[14])), "r"(__float_as_uint(v[15]))
        : "memory");
}
__device__ __forceinline__ void tmem_st8(unsigned addr, const float (&v)[8]) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};\n" ::"r"(addr),
                 "r"(__float_as_uint(v[0])), "r"(__float_as_uint(v[1])), "r"(__float_as_uint(v[2])),
                 "r"(__float_as_uint(v[3])), "r"(__float_as_uint(v[4])), "r"(__float_as_uint(v[5])),
                 "r"(__float_as_uint(v[6])), "r"(__float_as_uint(v[7]))
                 : "memory");
}
__device__ __forceinline__ void tmem_st16_zero(unsigned addr) {
    const unsigned z = 0u;
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1};\n" ::
            "r"(addr), "r"(z)
        : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;\n" ::: "memory"); }

// x = hi + lo with hi the nearest TF32 (10-bit mantissa, ties away from zero) and lo the remainder (the MMA truncates it to
// TF32).  hi is what cvt.rna.tf32.f32 returns for finite x - half an ulp of the short mantissa added to the magnitude, the
// low 13 bits cleared - in two integer instructions: the cvt compiles to four (it guards inf / nan), and the expanding
// warps of the tensor-core kernels, which split every operand element, are instruction-bound (ncu: gradw_ns 845 M warp
// instructions per launch; gradw_ts workers busy 83 % of the kernel).  inf stays inf, nan stays nan.
__device__ __forceinline__ void split_tf32(float x, float &hi, float &lo) {
    hi = __uint_as_float((__float_as_uint(x) + 0x1000u) & 0xffffe000u);
    lo = x - hi;
}

}  // namespace tc
}  // namespace tnmf
