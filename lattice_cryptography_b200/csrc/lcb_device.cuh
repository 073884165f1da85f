// lcb_device.cuh — device primitives shared by the lcb200 kernels (sm_100a).
//
//   * 32-bit modular arithmetic for q < 2^16 on the integer pipes: Shoup multiplication by
//     precomputed constants (IMAD.HI + 2 IMAD), Barrett reduction, lazy (unreduced) butterflies.
//   * d = 256 negacyclic NTT: one polynomial per HALF-WARP (16 lanes x 16 coefficients):
//     stages 1-4 and 5-8 run in registers, with ONE conflict-free transposition through shared
//     memory in between.  Stage 1-4 twiddles are warp-uniform (kernel-parameter constant bank),
//     stage 5-8 twiddles are 15 per-lane register pairs.
//   * Keccak-f[1600] with the state in registers (one SHAKE256 stream per thread).
//
// Replaces lattice_algebra's ntt()/cent()/Polynomial arithmetic and binary_digest() (restated in
// oracle/lattice_algebra/__init__.py).  The reference transform is a 2d-point cyclic NTT of the
// zero-padded polynomial; this one is the d-point negacyclic NTT, which yields the same
// coefficient representations (parity level L1) with half the work.
#pragma once
#include <cstdint>

#include <cuda_runtime.h>

// Checked build (make CHECKED=1 -> liblcb200_checked.so): every hand-rolled guard of a global access asserts the
// range it is about to touch.  compute-sanitizer is not available on the GPU pool (profiles/sanitizer_r2.txt), so
// this build plus tests/test_gpu_checked.py stands in for memcheck.  A failed check traps the kernel: the call
// returns LCB_ERR_CUDA ("device-side assert").
#ifdef LCB_CHECKED
#include <cassert>
#define LCB_CHECK(cond) assert(cond)
#else
#define LCB_CHECK(cond) ((void)0)
#endif

namespace lcb {

constexpr int D = 256;            // ring degree handled by the fast path
constexpr int LOGD = 8;
constexpr int LANES = 16;         // lanes per polynomial
constexpr int EPT = 16;           // coefficients per lane
constexpr int XROW = 20;          // padded row pitch (words) of the transposition buffer
constexpr int XHALF = 336;        // words per half-warp buffer: 16 rows * 20 + 16 (bank offset)
constexpr int XWARP = 2 * XHALF;  // words per warp

// Modulus constants; passed BY VALUE as a kernel parameter so they live in the constant bank.
struct ModQ {
    uint32_t zero;        // always 0, but opaque to the compiler: turns `a + b` into a 3-input IADD3 (ALU pipe)
                          // where ptxas would otherwise pick IMAD.IADD and load the FMA-heavy pipe further.
                          // Measured on k_verify (2^20 verifies): 5.46 ms with it in stages 1-4 and 5-8,
                          // 5.60 / 5.61 ms with it in only one group, 5.74 ms without.
    uint32_t q, negq;
    uint32_t barrett;     // floor((2^32-1)/q)
    uint32_t cq;          // least multiple of q >= 32768: makes any int16 input non-negative
    uint32_t cq2;         // least multiple of q >= 65536 + 2q: bound for u16-derived lazy values
    uint32_t half;        // (q-1)/2
    uint32_t dinv, dinv_s;  // d^-1 mod q and its Shoup companion
    uint32_t q4;          // 4q: positivity offset of the FP32-assisted butterflies
    uint32_t in_off;      // cq + 26 q + FP_BIAS: raw int16 coefficient -> biased lazy value that stays non-negative
                          // through eight offset-free butterfly stages (ntt_fwd_256_fp)
    uint32_t in_off_q4;   // (unused since the two-stage butterflies; kept so that the parameter layout is stable)
    uint32_t bias_mod_q;  // FP_BIAS mod q
    int32_t z1c;          // zetas[1] (the stage-1 twiddle) as a centred residue, |z1c| < 2^15
    uint32_t k1;          // least multiple of q >= 2^30 + 2^15: offset of the reduction-free first stage
    // exact divisibility test for the final comparison of k_verify: for odd q, a 64-bit x is a multiple of q iff
    // x * q^-1 mod 2^64 <= floor((2^64 - 1) / q) (multiplication by q^-1 permutes the residues mod 2^64 and sends
    // m * q to m) - three multiplies and a compare instead of three Barrett rounds and two conditional subtractions
    uint32_t qinv_lo, qinv_hi;    // q^-1 mod 2^64
    uint32_t dlim_lo, dlim_hi;    // floor((2^64 - 1) / q)
    uint32_t kq18;                // least multiple of q >= 2^18: keeps acc - (rhs + corr) non-negative
    uint32_t kw0;                 // (0x4B400000 + 2) * q mod 2^32: constant part of the FP32-assisted twiddle offset kw
};

// Warp-uniform twiddles of stages 1..4 (zeta index k = 1..15), forward and inverse.
struct StageConst {
    uint32_t w[16], ws[16], iw[16], iws[16];
};

// Per-lane twiddles of stages 5..8: [0] stage 5, [1..2] stage 6, [3..6] stage 7, [7..14] stage 8.
struct LaneTw {
    uint32_t w[15], ws[15];
};

// ---- FP32-assisted butterflies (forward transform of k_verify) -----------------------------------
// IMAD.HI issues at a quarter of the IMAD rate on sm_100 (tools/pipe_bench.cu: 30 vs 63 thread-instr/clk/SM),
// so the quotient estimate of a twiddle multiplication is taken from the FP32 pipe instead, where an FFMA
// is full rate and can issue beside the IMADs.  Lazy values r < 2^23 are carried BIASED, b = r + 0x4B000000:
// the same 32 bits read as the float 2^23 + r, so no conversion instruction exists at all.
//   qf  = fma(as_float(yb), w/q, 1.5*2^23 - 2^23*(w/q))        = 1.5*2^23 + round(y*w/q) (+-1.13)
//   t   = yb*w + kw                                            kw = (0x4B400000 + 2)*q - 0x4B000000*w  (mod 2^32)
//   T   = as_uint(qf)*(-q) + t  =  y*w - qhat*q + 2q           in (0.87 q, 3.13 q)
// One FFMA + two IMAD per multiplication instead of IMAD.HI + two IMAD; butterflies add at most 4q per stage.
constexpr uint32_t FP_BIAS = 0x4B000000u;

struct StageConstF {            // warp-uniform stages 1..4, zeta index k = 1..15 (kernel-parameter constant bank)
    uint32_t w[16];
    float wq[16], cst[16];
    uint32_t kw[16];
};

struct LaneTwF {                // per-lane stages 5..8, same indexing as LaneTw
    uint32_t w[15];
    float wq[15], cst[15];
    uint32_t kw[15];
    __device__ __forceinline__ void get(int k, uint32_t& w_, float& wq_, float& cst_, uint32_t& kw_) const {
        w_ = w[k]; wq_ = wq[k]; cst_ = cst[k]; kw_ = kw[k];
    }
};
// The same per-lane twiddles read from a shared-memory row at every use (frees 60 registers per thread), in two forms:
//   LaneTwFShared   {w, wq, cst, kw}: one LDS.128 per twiddle - four shared-memory wavefronts per warp, no arithmetic;
//   LaneTwFShared2  {w, wq}: one LDS.64 (two wavefronts); cst = 1.5*2^23 - 2^23*(w/q) and kw = (0x4B400000 + 2) q -
//                   0x4B000000 w are re-derived with one FFMA and one IMAD - bit-identical to the table values (the FFMA
//                   rounds the same real number once; the IMAD is exact mod 2^32).
// Which one wins depends on what binds the kernel (measured, round 2): k_sign sat at 86 % of the L1/shared-memory
// pipeline with 31 twiddle rows per polynomial as 63 % of its wavefronts (mio-throttle + short-scoreboard = 33 % of the
// warp samples) and gains 4.6 % from the short rows (6.36 -> 6.07 ms per 2^20); k_verify (15 rows per polynomial, 80 % of
// the pipeline but 71 % issue-active) loses 5 % to the 30 extra instructions per row (4.20 -> 4.42 ms) and keeps the long rows
// (re-tried on the 512-thread form, 89 % of the pipeline and 77 % issue-active: 3.87 -> 4.13 ms, still a loss).
struct LaneTwFShared {
    const uint4* row;
    __device__ __forceinline__ void get(int k, uint32_t& w_, float& wq_, float& cst_, uint32_t& kw_) const {
        const uint4 v = row[k];
        w_ = v.x; wq_ = __uint_as_float(v.y); cst_ = __uint_as_float(v.z); kw_ = v.w;
    }
};
struct LaneTwFShared2 {
    const uint2* row;
    uint32_t kw0;            // (0x4B400000 + 2) * q mod 2^32
    __device__ __forceinline__ void get(int k, uint32_t& w_, float& wq_, float& cst_, uint32_t& kw_) const {
        const uint2 v = row[k];
        w_ = v.x; wq_ = __uint_as_float(v.y);
        cst_ = __fmaf_rn(wq_, -8388608.0f, 12582912.0f);
        kw_ = w_ * (0u - FP_BIAS) + kw0;
    }
};

// Device-resident tables of one ctx.
struct NttTables {
    float f_wq[256], f_cst[256];   // FP32-assisted forward twiddles (see StageConstF)
    uint32_t f_kw[256];
    uint32_t w[256], ws[256];      // zetas[k] = psi^bitrev8(k) and Shoup companions
    uint32_t iw[256], iws[256];    // zetas[k]^-1
    uint32_t pw[512], pws[512];    // psi^e, e in [0, 512): NTT image of monomials (BKLM)
    uint16_t oddexp[256];          // 2*bitrev8(p)+1: exponent of the evaluation point of slot p
    // FP32-assisted INVERSE transform (ntt_inv_256_fp): per lane 31 entries {w, w/q, cst, kw}: [0] half 16,
    // [1..2] half 32, [3..6] half 64, [7..14] half 128 (twiddle omega^-((256/half) j), j = lane + 16 (jj mod half/16)),
    // [15..30] the closing twist psi^-i d^-1, i = lane + 16 jj
    uint4 inv_lane[16][31];
};

__device__ __forceinline__ uint32_t shoup_mul(uint32_t a, uint32_t w, uint32_t ws, const ModQ& m) {
    // a any 32-bit value, w < q, ws = floor(w * 2^32 / q)  ->  a*w mod q in [0, 2q)
    uint32_t hi = __umulhi(a, ws);
    return a * w + hi * m.negq;
}

__device__ __forceinline__ uint32_t barrett_lazy(uint32_t x, const ModQ& m) {
    // x any 32-bit value -> x mod q in [0, 2q): with 2^32 - 1 = barrett q + s (s < q) and x = Q q + R, the estimate is
    // short by two only if R barrett + 2^32 < Q (1 + s), and Q (1 + s) < 2^32 (1 + s) / q <= 2^32
    // (tests/test_verify_tc_limbs_cpu.py checks the inputs of k_verify_tc's limb reduction exhaustively)
    uint32_t hi = __umulhi(x, m.barrett);
    return x + hi * m.negq;
}

__device__ __forceinline__ uint32_t csub(uint32_t x, uint32_t q) { return x >= q ? x - q : x; }

__device__ __forceinline__ uint32_t barrett_full(uint32_t x, const ModQ& m) {
    // floor((2^32-1)/q) underestimates the quotient by at most 1 (barrett_lazy); the second subtraction never fires
    return csub(csub(barrett_lazy(x, m), m.q), m.q);
}

__device__ __forceinline__ uint32_t mulmod_full(uint32_t a, uint32_t b, const ModQ& m) {
    // a, b < 2^16 -> a*b mod q in [0, q)
    return barrett_full(a * b, m);
}

__device__ __forceinline__ uint32_t reduce64(uint64_t acc, const ModQ& m) {
    // acc < 2^54 -> acc mod q in [0, q)   (q < 2^16): three 12-bit-shifted Barrett steps
    uint32_t r = barrett_full((uint32_t)(acc >> 24), m);
    r = barrett_full((r << 12) | ((uint32_t)(acc >> 12) & 0xFFFu), m);
    return barrett_full((r << 12) | ((uint32_t)acc & 0xFFFu), m);
}

__device__ __forceinline__ bool divisible_by_q(uint64_t x, const ModQ& m) {
    const uint64_t qinv = ((uint64_t)m.qinv_hi << 32) | m.qinv_lo, lim = ((uint64_t)m.dlim_hi << 32) | m.dlim_lo;
    return x * qinv <= lim;
}

__device__ __forceinline__ int32_t center(uint32_t r, const ModQ& m) {
    // r in [0, q) -> centred residue
    return r > m.half ? (int32_t)r - (int32_t)m.q : (int32_t)r;
}

__device__ __forceinline__ void load_lane_tw(LaneTw& t, const uint32_t* __restrict__ w,
                                             const uint32_t* __restrict__ ws, int lane) {
    t.w[0] = __ldg(w + 16 + lane);
    t.ws[0] = __ldg(ws + 16 + lane);
#pragma unroll
    for (int i = 0; i < 2; ++i) { t.w[1 + i] = __ldg(w + 32 + 2 * lane + i); t.ws[1 + i] = __ldg(ws + 32 + 2 * lane + i); }
#pragma unroll
    for (int i = 0; i < 4; ++i) { t.w[3 + i] = __ldg(w + 64 + 4 * lane + i); t.ws[3 + i] = __ldg(ws + 64 + 4 * lane + i); }
#pragma unroll
    for (int i = 0; i < 8; ++i) { t.w[7 + i] = __ldg(w + 128 + 8 * lane + i); t.ws[7 + i] = __ldg(ws + 128 + 8 * lane + i); }
}

// ---- transposition between the two register layouts -------------------------------------------
// layout A: r[j] = x[lane + 16 j]      (strides 128..16 are inside a lane)
// layout B: r[m] = x[16 lane + m]      (strides 8..1 are inside a lane)
__device__ __forceinline__ void xpose_a_to_b(uint32_t (&r)[EPT], uint32_t* xb, int lane) {
#pragma unroll
    for (int j = 0; j < EPT; ++j) xb[XROW * j + lane] = r[j];
    __syncwarp();
#pragma unroll
    for (int g = 0; g < 4; ++g) {
        uint4 v = *reinterpret_cast<const uint4*>(xb + XROW * lane + 4 * g);
        r[4 * g] = v.x; r[4 * g + 1] = v.y; r[4 * g + 2] = v.z; r[4 * g + 3] = v.w;
    }
    __syncwarp();
}

__device__ __forceinline__ void xpose_b_to_a(uint32_t (&r)[EPT], uint32_t* xb, int lane) {
#pragma unroll
    for (int g = 0; g < 4; ++g)
        *reinterpret_cast<uint4*>(xb + XROW * lane + 4 * g) = make_uint4(r[4 * g], r[4 * g + 1], r[4 * g + 2], r[4 * g + 3]);
    __syncwarp();
#pragma unroll
    for (int j = 0; j < EPT; ++j) r[j] = xb[XROW * j + lane];
    __syncwarp();
}

// ---- forward negacyclic NTT, Cooley-Tukey, natural order in (layout A) -> bit-reversed out (layout B)
// input values < 2^17; every stage adds < 2q, so outputs are < 2^17 + 16 q < 2^21 (lazy).
__device__ __forceinline__ void ntt_fwd_256(uint32_t (&r)[EPT], const ModQ& m, const StageConst& sc,
                                            const LaneTw& tw, uint32_t* xb, int lane) {
    const uint32_t q2 = 2 * m.q;
#pragma unroll
    for (int s = 1; s <= 4; ++s) {
        const int len = 8 >> (s - 1);
#pragma unroll
        for (int j = 0; j < EPT; ++j) {
            if (j & len) continue;
            const int k = (1 << (s - 1)) + (j >> (5 - s));
            uint32_t t = shoup_mul(r[j + len], sc.w[k], sc.ws[k], m);
            r[j + len] = r[j] + q2 - t;
            r[j] = r[j] + t + m.zero;
        }
    }
    xpose_a_to_b(r, xb, lane);
#pragma unroll
    for (int s = 5; s <= 8; ++s) {
        const int len = 256 >> s;
        const int base = (1 << (s - 5)) - 1;
#pragma unroll
        for (int j = 0; j < EPT; ++j) {
            if (j & len) continue;
            const int k = base + (j >> (9 - s));
            uint32_t t = shoup_mul(r[j + len], tw.w[k], tw.ws[k], m);
            r[j + len] = r[j] + q2 - t;
            r[j] = r[j] + t + m.zero;
        }
    }
}

// Same transform for RAW centred int16 coefficients (any value in [-2^15, 2^15)): the first stage needs
// no modular reduction at all, because |x * z1c| < 2^30 fits a word: X' = X + z1c*Y + k1, Y' = X - z1c*Y + k1
// with k1 = 0 mod q.  One IMAD instead of IMAD.HI + 2 IMAD per first-stage butterfly, and no input
// offset.  Outputs are < 2^31 + 2^16 + 14 q < 2^32 (lazy); 64-bit row-vector accumulators stay < 2^54.
__device__ __forceinline__ void ntt_fwd_256_raw(const int (&x)[EPT], uint32_t (&r)[EPT], const ModQ& m,
                                                const StageConst& sc, const LaneTw& tw, uint32_t* xb, int lane) {
    const uint32_t q2 = 2 * m.q;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        const int t = x[j + 8] * m.z1c;
        r[j] = (uint32_t)(x[j] + t) + m.k1;
        r[j + 8] = (uint32_t)(x[j] - t) + m.k1;
    }
#pragma unroll
    for (int s = 2; s <= 4; ++s) {
        const int len = 8 >> (s - 1);
#pragma unroll
        for (int j = 0; j < EPT; ++j) {
            if (j & len) continue;
            const int k = (1 << (s - 1)) + (j >> (5 - s));
            uint32_t t = shoup_mul(r[j + len], sc.w[k], sc.ws[k], m);
            r[j + len] = r[j] + q2 - t;
            r[j] = r[j] + t + m.zero;
        }
    }
    xpose_a_to_b(r, xb, lane);
#pragma unroll
    for (int s = 5; s <= 8; ++s) {
        const int len = 256 >> s;
        const int base = (1 << (s - 5)) - 1;
#pragma unroll
        for (int j = 0; j < EPT; ++j) {
            if (j & len) continue;
            const int k = base + (j >> (9 - s));
            uint32_t t = shoup_mul(r[j + len], tw.w[k], tw.ws[k], m);
            r[j + len] = r[j] + q2 - t;
            r[j] = r[j] + t + m.zero;
        }
    }
}

__device__ __forceinline__ void load_lane_tw_f(LaneTwF& t, const NttTables* __restrict__ tab, int lane) {
    auto put = [&](int dst, int k) {
        t.w[dst] = __ldg(tab->w + k);
        t.wq[dst] = __ldg(tab->f_wq + k);
        t.cst[dst] = __ldg(tab->f_cst + k);
        t.kw[dst] = __ldg(tab->f_kw + k);
    };
    put(0, 16 + lane);
#pragma unroll
    for (int i = 0; i < 2; ++i) put(1 + i, 32 + 2 * lane + i);
#pragma unroll
    for (int i = 0; i < 4; ++i) put(3 + i, 64 + 4 * lane + i);
#pragma unroll
    for (int i = 0; i < 8; ++i) put(7 + i, 128 + 8 * lane + i);
}

// yb biased (y < 2^22)  ->  y*w mod q + {0,1,2,3}q, in (0.87 q, 3.13 q), NOT biased
__device__ __forceinline__ uint32_t fp_mul(uint32_t yb, uint32_t w, float wq, float cst, uint32_t kw, const ModQ& m) {
    const float qf = __fmaf_rn(__uint_as_float(yb), wq, cst);
    const uint32_t t = yb * w + kw;
    return __float_as_uint(qf) * m.negq + t;
}

// Forward transform of RAW centred int16 coefficients with FP32-assisted butterflies, two stages at a time.
// A pair of Cooley-Tukey stages acts on quadruples (a, b, c, d) = r[i], r[i+h], r[i+2h], r[i+3h]:
//     first stage   a' = a + Tc, c' = a - Tc, b' = b + Td, d' = b - Td            (Tc = c*w, Td = d*w)
//     second stage  a'' = a' + T1, b'' = a' - T1, c'' = c' + T2, d'' = c' - T2    (T1 = b'*w0, T2 = d'*w1)
// Only b' and d' are multiplied again, so a' and c' are never formed: a'' = a + Tc + T1, b'' = a + Tc - T1,
// c'' = a - Tc + T2, d'' = a - Tc - T2 are four 3-input adds - 6 adds per quadruple instead of 8, 18 instructions instead
// of 20 (round 2; k_verify 4.25 -> see DESIGN.md).  A 3-input add has no slot for the "+4q" that kept differences
// positive, so positivity comes from the INPUT offset instead: products are T in (0.87 q, 3.13 q), every stage moves a
// value by at most 3.13 q either way, and inputs enter as x + cq + 26 q (in_off): after eight stages values lie in
// (0.9 q, cq + 2^15 + 52 q) - non-negative, and below 2^22 for every q < 2^16, where the FP32 quotient estimate is exact
// to +-1.  Values stay biased throughout; outputs are UNBIASED lazy values < 2^22 PLUS FP_BIAS in layout B.
// x + y + z and friends as ONE IADD3 each: two dependent PTX adds in an asm block (ptxas fuses them; written in C++ the
// compiler regroups the four sums of a quadruple around their common a + tc / a - tc and is back at eight adds)
__device__ __forceinline__ uint32_t add3_pp(uint32_t x, uint32_t y, uint32_t z) {
    uint32_t o;
    asm("{ .reg .u32 t; add.u32 t, %1, %2; add.u32 %0, t, %3; }" : "=r"(o) : "r"(x), "r"(y), "r"(z));
    return o;
}
__device__ __forceinline__ uint32_t add3_pm(uint32_t x, uint32_t y, uint32_t z) {   // x + y - z
    uint32_t o;
    asm("{ .reg .u32 t; add.u32 t, %1, %2; sub.u32 %0, t, %3; }" : "=r"(o) : "r"(x), "r"(y), "r"(z));
    return o;
}
__device__ __forceinline__ uint32_t add3_mm(uint32_t x, uint32_t y, uint32_t z) {   // x - y - z
    uint32_t o;
    asm("{ .reg .u32 t; sub.u32 t, %1, %2; sub.u32 %0, t, %3; }" : "=r"(o) : "r"(x), "r"(y), "r"(z));
    return o;
}

// RAW = true: a and b arrive without the input offset `off` (it joins a's explicit add and b's 3-input adds)
template <bool RAW, typename GET>
__device__ __forceinline__ void fp_quad(uint32_t& a, uint32_t& b, uint32_t& c, uint32_t& d, int kA, int kB0, int kB1,
                                        const ModQ& m, GET&& get, uint32_t off = 0) {
    uint32_t w_, kw_;
    float wq_, cst_;
    get(kA, w_, wq_, cst_, kw_);
    const uint32_t tc = fp_mul(c, w_, wq_, cst_, kw_, m), td = fp_mul(d, w_, wq_, cst_, kw_, m);
    uint32_t b1, d1;
    if (RAW) {
        b1 = add3_pp(b, off, td);
        d1 = add3_pm(b, off, td);
        a = a + off + m.zero;
    } else {
        b1 = b + td + m.zero;
        d1 = b - td + m.zero;
    }
    get(kB0, w_, wq_, cst_, kw_);
    const uint32_t t1 = fp_mul(b1, w_, wq_, cst_, kw_, m);
    get(kB1, w_, wq_, cst_, kw_);
    const uint32_t t2 = fp_mul(d1, w_, wq_, cst_, kw_, m);
    // grouped so that no two results share a subexpression
    const uint32_t na = add3_pp(a, t1, tc), nb = add3_pm(a, tc, t1), nc = add3_pm(a, t2, tc), nd = add3_mm(a, t2, tc);
    a = na; b = nb; c = nc; d = nd;
}

template <typename TW>
__device__ __forceinline__ void ntt_fwd_256_fp(const int (&x)[EPT], uint32_t (&r)[EPT], const ModQ& m,
                                               const StageConstF& sc, const TW& tw, uint32_t* xb, int lane) {
    auto uni = [&](int k, uint32_t& w_, float& wq_, float& cst_, uint32_t& kw_) {
        w_ = sc.w[k]; wq_ = sc.wq[k]; cst_ = sc.cst[k]; kw_ = sc.kw[k];
    };
    auto per_lane = [&](int k, uint32_t& w_, float& wq_, float& cst_, uint32_t& kw_) { tw.get(k, w_, wq_, cst_, kw_); };
    // stages 1 + 2 (distances 8, 4): the inputs take their offset on the way in
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        r[j] = (uint32_t)x[j];
        r[j + 4] = (uint32_t)x[j + 4];
        r[j + 8] = (uint32_t)x[j + 8] + m.in_off + m.zero;
        r[j + 12] = (uint32_t)x[j + 12] + m.in_off + m.zero;
        fp_quad<true>(r[j], r[j + 4], r[j + 8], r[j + 12], 1, 2, 3, m, uni, m.in_off);
    }
    // stages 3 + 4 (distances 2, 1)
#pragma unroll
    for (int g = 0; g < 4; ++g) fp_quad<false>(r[4 * g], r[4 * g + 1], r[4 * g + 2], r[4 * g + 3], 4 + g, 8 + 2 * g, 9 + 2 * g, m, uni);
    xpose_a_to_b(r, xb, lane);
    // stages 5 + 6, 7 + 8: the same index pattern on the per-lane twiddles (LaneTwF indexing = stage index - 1)
#pragma unroll
    for (int j = 0; j < 4; ++j) fp_quad<false>(r[j], r[j + 4], r[j + 8], r[j + 12], 0, 1, 2, m, per_lane);
#pragma unroll
    for (int g = 0; g < 4; ++g) fp_quad<false>(r[4 * g], r[4 * g + 1], r[4 * g + 2], r[4 * g + 3], 3 + g, 7 + 2 * g, 8 + 2 * g, m, per_lane);
    // outputs stay BIASED (r + FP_BIAS): the caller's multiply-accumulate removes the bias once per slot
}

// ---- inverse, Gentleman-Sande, bit-reversed in (layout B) -> natural order out (layout A), UNSCALED
// (multiply by d^-1 afterwards).  Inputs < b0 (a multiple of q); outputs < 256 * b0.
__device__ __forceinline__ void ntt_inv_256(uint32_t (&r)[EPT], const ModQ& m, const StageConst& sc,
                                            const LaneTw& itw, uint32_t* xb, int lane, uint32_t b0) {
    uint32_t b = b0;
#pragma unroll
    for (int s = 8; s >= 5; --s) {
        const int len = 256 >> s;
        const int base = (1 << (s - 5)) - 1;
#pragma unroll
        for (int j = 0; j < EPT; ++j) {
            if (j & len) continue;
            const int k = base + (j >> (9 - s));
            uint32_t x = r[j], y = r[j + len];
            r[j] = x + y;
            r[j + len] = shoup_mul(x + b - y, itw.w[k], itw.ws[k], m);
        }
        b <<= 1;
    }
    xpose_b_to_a(r, xb, lane);
#pragma unroll
    for (int s = 4; s >= 1; --s) {
        const int len = 8 >> (s - 1);
#pragma unroll
        for (int j = 0; j < EPT; ++j) {
            if (j & len) continue;
            const int k = (1 << (s - 1)) + (j >> (5 - s));
            uint32_t x = r[j], y = r[j + len];
            r[j] = x + y;
            r[j + len] = shoup_mul(x + b - y, sc.iw[k], sc.iws[k], m);
        }
        b <<= 1;
    }
}

// ---- inverse with FP32-assisted butterflies (k_sign) ---------------------------------------------------------
// The Gentleman-Sande inverse above multiplies AFTER the subtraction: its operands double from stage to stage
// (2^17 -> 2^25), out of reach of the FP32 quotient estimate (exact below 2^22), so it stays on Shoup multiplications
// whose IMAD.HI issues at a quarter of the IMAD rate - k_sign was bound by the FMA-heavy pipe (96 IMAD.HI per row).
// The slot order of this library IS the bit-reversed order of the 256-point cyclic transform of b_i = a_i psi^i
// (slot p holds a(psi^(2 bitrev(p) + 1)) = DFT_omega(b)[bitrev(p)], omega = psi^2), so the inverse can just as well be
// the decimation-in-time form: Cooley-Tukey butterflies (u + w v, u - w v) with twiddles omega^-j, half = 1, 2, ..
// 128, natural order out, followed by the twist a_i = A_i psi^-i d^-1 - which replaces the d^-1 scaling, so it is free.
// Multiplying BEFORE the add keeps growth additive (+4q per stage): the FP32-assisted multiplication of the forward
// transform applies (one FFMA + two IMAD, no IMAD.HI).  Butterflies with w = 1 are plain adds in stages 1-3 (doubling
// three times is affordable: 2^16 + 2q -> < 2^21); from stage 4 on w = 1 is multiplied like any other twiddle.
// 50 multiplications + 16 for the twist instead of 64 + 16.
// in : layout B, BIASED lazy values < 2^16 + 2q + FP_BIAS;  out: layout A, unbiased twisted values in (0.87 q, 3.13 q)
template <typename TW>
__device__ __forceinline__ void ntt_inv_256_fp(uint32_t (&r)[EPT], const ModQ& m, const StageConstF& isc, const TW& tw,
                                               uint32_t* xb, int lane) {
#pragma unroll
    for (int s = 1; s <= 4; ++s) {
        const int half = 1 << (s - 1);
        const uint32_t off = FP_BIAS + (m.q4 << (s - 1));       // 4q, 8q, 16q: at least the bound of the stage's inputs
#pragma unroll
        for (int j = 0; j < EPT; ++j) {
            if (j & half) continue;
            const int e = j & (half - 1);
            if (e == 0 && s <= 3) {
                const uint32_t u = r[j], v = r[j + half];
                r[j] = u + v - FP_BIAS;
                r[j + half] = u - v + off;
            } else {
                const int k = half + e;
                const uint32_t t = fp_mul(r[j + half], isc.w[k], isc.wq[k], isc.cst[k], isc.kw[k], m);
                r[j + half] = r[j] + m.q4 - t;
                r[j] = r[j] + t + m.zero;
            }
        }
    }
    xpose_b_to_a(r, xb, lane);
#pragma unroll
    for (int s = 5; s <= 8; ++s) {
        const int h16 = 1 << (s - 5);
#pragma unroll
        for (int j = 0; j < EPT; ++j) {
            if (j & h16) continue;
            uint32_t w_, kw_;
            float wq_, cst_;
            tw.get((h16 - 1) + (j & (h16 - 1)), w_, wq_, cst_, kw_);
            const uint32_t t = fp_mul(r[j + h16], w_, wq_, cst_, kw_, m);
            r[j + h16] = r[j] + m.q4 - t;
            r[j] = r[j] + t + m.zero;
        }
    }
#pragma unroll
    for (int j = 0; j < EPT; ++j) {
        uint32_t w_, kw_;
        float wq_, cst_;
        tw.get(15 + j, w_, wq_, cst_, kw_);
        r[j] = fp_mul(r[j], w_, wq_, cst_, kw_, m);
    }
}

// value in (0, 4q) congruent to the coefficient -> centred coefficient
__device__ __forceinline__ int32_t center_lazy4(uint32_t t, const ModQ& m) {
    const uint32_t q2 = 2 * m.q;
    t = min(t, t - q2);          // unsigned wrap-around: subtracts only when t >= 2q
    t = min(t, t - m.q);
    return center(t, m);
}

// final scaling of an unscaled inverse transform value -> centred coefficient
__device__ __forceinline__ int32_t finish_coef(uint32_t v, const ModQ& m) {
    return center(csub(shoup_mul(v, m.dinv, m.dinv_s, m), m.q), m);
}

// ---- 16 consecutive uint16 <-> registers (NTT-form rows, 32 B per lane, 512 B per half-warp)
__device__ __forceinline__ void load_u16x16(uint32_t (&r)[EPT], const uint16_t* __restrict__ p) {
    const uint4* v = reinterpret_cast<const uint4*>(p);
    uint4 a = __ldg(v), b = __ldg(v + 1);
    uint32_t w[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
#pragma unroll
    for (int i = 0; i < 8; ++i) { r[2 * i] = w[i] & 0xFFFFu; r[2 * i + 1] = w[i] >> 16; }
}

__device__ __forceinline__ void store_u16x16(uint16_t* __restrict__ p, const uint32_t (&r)[EPT]) {
    uint32_t w[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) w[i] = (r[2 * i] & 0xFFFFu) | (r[2 * i + 1] << 16);
    uint4* v = reinterpret_cast<uint4*>(p);
    v[0] = make_uint4(w[0], w[1], w[2], w[3]);
    v[1] = make_uint4(w[4], w[5], w[6], w[7]);
}

// ---- Keccak-f[1600] -----------------------------------------------------------------------------
// State as 25 (lo, hi) pairs of 32-bit registers; written so that ptxas emits exactly the minimum:
// per round 122 LOP3 (5-way column parities as two xor3; theta applied as a ^ C[x-1] ^ rotl(C[x+1],1)
// in one LOP3 without forming D; chi as one LOP3 each) and 58 SHF (funnel shifts for rho and the
// theta rotation), no register moves.  Measured 4.28 Gperm/s on B200 = the ALU-pipe issue limit
// (64 lanes/clk/SM) for 24 x 180 instructions (tools/keccak_bench2.cu; moving rotations onto the FMA
// pipe as IMAD.WIDE/IMAD.HI multiplies by 2^n was measured there too and loses).
#define LCB_KECCAK_RC_INIT                                                                           \
    {0x0000000000000001ULL, 0x0000000000008082ULL, 0x800000000000808aULL, 0x8000000080008000ULL,     \
     0x000000000000808bULL, 0x0000000080000001ULL, 0x8000000080008081ULL, 0x8000000000008009ULL,     \
     0x000000000000008aULL, 0x0000000000000088ULL, 0x0000000080008009ULL, 0x000000008000000aULL,     \
     0x000000008000808bULL, 0x800000000000008bULL, 0x8000000000008089ULL, 0x8000000000008003ULL,     \
     0x8000000000008002ULL, 0x8000000000000080ULL, 0x000000000000800aULL, 0x800000008000000aULL,     \
     0x8000000080008081ULL, 0x8000000000008080ULL, 0x0000000080000001ULL, 0x8000000080008008ULL}

__host__ __device__ constexpr int keccak_pi(int i) {
    // lane index i = x + 5y;  (x, y) -> (y, 2x + 3y)
    return (i / 5) + 5 * ((2 * (i % 5) + 3 * (i / 5)) % 5);
}

struct KeccakState {
    uint32_t lo[25], hi[25];
};

__device__ __forceinline__ uint32_t lop_xor3(uint32_t a, uint32_t b, uint32_t c) {
    uint32_t d;
    asm("lop3.b32 %0, %1, %2, %3, 0x96;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
    return d;
}
__device__ __forceinline__ uint32_t lop_chi(uint32_t a, uint32_t b, uint32_t c) {   // a ^ (~b & c)
    uint32_t d;
    asm("lop3.b32 %0, %1, %2, %3, 0xD2;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
    return d;
}
template <int N>
__device__ __forceinline__ void rotl64_pair(uint32_t lo, uint32_t hi, uint32_t& olo, uint32_t& ohi) {
    constexpr unsigned S = (unsigned)(N & 31);
    if (N == 0) { olo = lo; ohi = hi; }
    else if (N < 32) { ohi = __funnelshift_l(lo, hi, S); olo = __funnelshift_l(hi, lo, S); }
    else if (N == 32) { olo = hi; ohi = lo; }
    else { ohi = __funnelshift_l(hi, lo, S); olo = __funnelshift_l(lo, hi, S); }
}
template <int I>
struct KeccakRhoPi {
    // theta folded into the rotation input: a ^ C[x-1] ^ rotl(C[x+1], 1) is ONE LOP3, so D is never formed
    __device__ static __forceinline__ void run(const KeccakState& s, const uint32_t (&clo)[5], const uint32_t (&chi)[5],
                                               const uint32_t (&rlo)[5], const uint32_t (&rhi)[5], KeccakState& b) {
        constexpr int R[25] = {0, 1, 62, 28, 27, 36, 44, 6, 55, 20, 3, 10, 43, 25, 39, 41, 45, 15, 21, 8, 18, 2, 61, 56, 14};
        constexpr int x = I % 5;
        rotl64_pair<R[I]>(lop_xor3(s.lo[I], clo[(x + 4) % 5], rlo[(x + 1) % 5]),
                          lop_xor3(s.hi[I], chi[(x + 4) % 5], rhi[(x + 1) % 5]), b.lo[keccak_pi(I)], b.hi[keccak_pi(I)]);
        KeccakRhoPi<I + 1>::run(s, clo, chi, rlo, rhi, b);
    }
};
template <>
struct KeccakRhoPi<25> {
    __device__ static __forceinline__ void run(const KeccakState&, const uint32_t (&)[5], const uint32_t (&)[5],
                                               const uint32_t (&)[5], const uint32_t (&)[5], KeccakState&) {}
};

__device__ __forceinline__ void keccak_f1600(KeccakState& s, const uint64_t* __restrict__ rc) {
#pragma unroll 2
    for (int round = 0; round < 24; ++round) {
        uint32_t clo[5], chi[5], rlo[5], rhi[5];
#pragma unroll
        for (int x = 0; x < 5; ++x) {
            clo[x] = lop_xor3(lop_xor3(s.lo[x], s.lo[x + 5], s.lo[x + 10]), s.lo[x + 15], s.lo[x + 20]);
            chi[x] = lop_xor3(lop_xor3(s.hi[x], s.hi[x + 5], s.hi[x + 10]), s.hi[x + 15], s.hi[x + 20]);
        }
#pragma unroll
        for (int x = 0; x < 5; ++x) rotl64_pair<1>(clo[x], chi[x], rlo[x], rhi[x]);
        KeccakState b;
        KeccakRhoPi<0>::run(s, clo, chi, rlo, rhi, b);
#pragma unroll
        for (int y = 0; y < 5; ++y)
#pragma unroll
            for (int x = 0; x < 5; ++x) {
                s.lo[x + 5 * y] = lop_chi(b.lo[x + 5 * y], b.lo[(x + 1) % 5 + 5 * y], b.lo[(x + 2) % 5 + 5 * y]);
                s.hi[x + 5 * y] = lop_chi(b.hi[x + 5 * y], b.hi[(x + 1) % 5 + 5 * y], b.hi[(x + 2) % 5 + 5 * y]);
            }
        const uint64_t c = rc[round];
        s.lo[0] ^= (uint32_t)c;
        s.hi[0] ^= (uint32_t)(c >> 32);
    }
}

// ---- Keccak-f[1600] on TWO adjacent lanes per sponge (bit-interleaved halves) ---------------------
// A kernel with few, long SHAKE streams (BKLM aggregation coefficients on 8 GPUs: 8,192 streams of 59,754
// permutations each; a single key generation) leaves most of the 592 warp schedulers without a warp when a
// sponge is one thread.  Here lane 2i holds the EVEN bits and lane 2i+1 the ODD bits of each of the 25 state
// words (32 bits of every 64-bit word): theta's parities, chi and iota act on bit positions independently, so
// they stay lane-local; a rotation by an even amount 2a is a 32-bit rotation by a of the own half, a rotation by
// an odd amount 2a+1 takes the PARTNER's half rotated by a (odd lane) or a+1 (even lane) - one SHFL.  Per round
// and lane: 61 LOP3 + 29 SHF (exactly half of the one-thread form's 122 + 58, so the ALU-pipe roofline per
// permutation is unchanged) + 17 SHFL (12 odd rho offsets + 5 for theta's rotl(C,1)).
struct KeccakHalf {
    uint32_t a[25];
};

// (even, odd) bit halves of a 64-bit word
__host__ __device__ __forceinline__ uint32_t keccak_even_bits(uint64_t x) {
    x &= 0x5555555555555555ULL;
    x = (x | (x >> 1)) & 0x3333333333333333ULL;
    x = (x | (x >> 2)) & 0x0F0F0F0F0F0F0F0FULL;
    x = (x | (x >> 4)) & 0x00FF00FF00FF00FFULL;
    x = (x | (x >> 8)) & 0x0000FFFF0000FFFFULL;
    x = (x | (x >> 16)) & 0x00000000FFFFFFFFULL;
    return (uint32_t)x;
}
__host__ __device__ __forceinline__ uint32_t keccak_half_of(uint64_t x, unsigned odd) { return keccak_even_bits(x >> odd); }

// Rotation amounts of the odd rho offsets (and of theta's rotl 1) differ by one between the two lanes of a pair:
// a + 1 on the even lane, a on the odd lane, a = offset >> 1.  The twelve distinct values are pinned in registers
// by keccak_half_rot_init (volatile asm: ptxas otherwise re-derives each one from SR_TID at every use - S2R + LOP3
// + IADD3, 15 % more ALU instructions per round).
struct KeccakHalfRot {
    uint32_t s[12];
};
__host__ __device__ constexpr int keccak_half_rot_slot(int a) {
    constexpr int A[12] = {0, 1, 7, 10, 12, 13, 19, 20, 21, 22, 27, 30};
    for (int i = 0; i < 12; ++i)
        if (A[i] == a) return i;
    return -1;
}
__device__ __forceinline__ void keccak_half_rot_init(KeccakHalfRot& r, unsigned odd) {
    constexpr int A[12] = {0, 1, 7, 10, 12, 13, 19, 20, 21, 22, 27, 30};
    const uint32_t up = 1u - odd;
#pragma unroll
    for (int i = 0; i < 12; ++i) asm volatile("add.u32 %0, %1, %2;" : "=r"(r.s[i]) : "r"(up), "r"((uint32_t)A[i]));
}

template <int I>
struct KeccakHalfRhoPi {
    __device__ static __forceinline__ void run(const KeccakHalf& s, const uint32_t (&c)[5], const uint32_t (&r1)[5],
                                               const KeccakHalfRot& rot, KeccakHalf& b) {
        constexpr int R[25] = {0, 1, 62, 28, 27, 36, 44, 6, 55, 20, 3, 10, 43, 25, 39, 41, 45, 15, 21, 8, 18, 2, 61, 56, 14};
        constexpr int x = I % 5;
        const uint32_t t = lop_xor3(s.a[I], c[(x + 4) % 5], r1[(x + 1) % 5]);
        if (R[I] == 0) b.a[keccak_pi(I)] = t;
        else if (R[I] % 2 == 0) b.a[keccak_pi(I)] = __funnelshift_l(t, t, R[I] / 2);
        else {
            static_assert(R[I] % 2 == 0 || keccak_half_rot_slot(R[I] / 2) >= 0, "rotation table");
            const uint32_t o = __shfl_xor_sync(0xFFFFFFFFu, t, 1);
            b.a[keccak_pi(I)] = __funnelshift_l(o, o, rot.s[keccak_half_rot_slot(R[I] / 2)]);
        }
        KeccakHalfRhoPi<I + 1>::run(s, c, r1, rot, b);
    }
};
template <>
struct KeccakHalfRhoPi<25> {
    __device__ static __forceinline__ void run(const KeccakHalf&, const uint32_t (&)[5], const uint32_t (&)[5],
                                               const KeccakHalfRot&, KeccakHalf&) {}
};

// rc = this lane's halves of the 24 round constants (even-bit halves on even lanes, odd-bit halves on odd lanes).
// All 32 lanes of the warp must be active and converged.
// Measured dead end (tools/agg_coefs_timing.py, round 2): fetching the partner's raw odd-rho words and parities up front
// and forming its theta-applied word locally (one dependent exchange per round instead of two, 5 more SHF) changes
// nothing at one warp per scheduler (173 vs 174 ms).  What a lone warp pays (tools/halfwarp_bench.cu): two cycles per
// ALU-pipe instruction, about half a cycle to one cycle per instruction of another pipe (LOP3 + IMAD 1:1 issue at 0.79
// per cycle; 90 LOP3 + 17 independent SHFL take 190 cycles), so the 90 LOP3/SHF of a round are a floor of 180 cycles
// and the SHFL, the round-constant load and loop control come on top - hence 12 rounds per loop body below.  Rotations
// moved to the FMA pipe (IMAD.HI + IMAD by 2^a, no ALU instruction) were measured too: 30.3 instead of 19.3 ms.
// Rounds per loop body.  A lone warp per scheduler (the regime this form exists for) pays every instruction that is not
// on the ALU pipe - loop control, the round-constant load - with issue cycles nothing else fills: 8,192 streams of 7,472
// permutations take 21.6 / 20.5 / 20.3 / 19.8 / 19.3 ms with 1 / 2 / 4 / 8 / 12 rounds per body; all 24 (2,660
// instructions, 43 KB) overflow the instruction cache: 33 ms (profiles/exp_r2_keccak_half_unroll.txt).
// The cooperative sampler shares its SM's instruction cache between this loop and the decoder warps: there 12 rounds
// per body cost 3.46 ms per single key generation against 2.81 / 2.74 / 2.75 ms with 2 / 4 / 6 - hence a template
// parameter: 12 in k_agg_coefs_il, 4 in k_sampler_coop.
template <int UNROLL>
__device__ __forceinline__ void keccak_f1600_half(KeccakHalf& s, const uint32_t* __restrict__ rc, const KeccakHalfRot& rot) {
#pragma unroll UNROLL
    for (int round = 0; round < 24; ++round) {
        uint32_t c[5], r1[5];
#pragma unroll
        for (int x = 0; x < 5; ++x) c[x] = lop_xor3(lop_xor3(s.a[x], s.a[x + 5], s.a[x + 10]), s.a[x + 15], s.a[x + 20]);
#pragma unroll
        for (int x = 0; x < 5; ++x) {                      // rotl64(C, 1): partner's half, rotated by 1 on even lanes
            const uint32_t o = __shfl_xor_sync(0xFFFFFFFFu, c[x], 1);
            r1[x] = __funnelshift_l(o, o, rot.s[0]);
        }
        KeccakHalf b;
        KeccakHalfRhoPi<0>::run(s, c, r1, rot, b);
#pragma unroll
        for (int y = 0; y < 5; ++y)
#pragma unroll
            for (int x = 0; x < 5; ++x)
                s.a[x + 5 * y] = lop_chi(b.a[x + 5 * y], b.a[(x + 1) % 5 + 5 * y], b.a[(x + 2) % 5 + 5 * y]);
        s.a[0] ^= rc[round];
    }
}

}  // namespace lcb
