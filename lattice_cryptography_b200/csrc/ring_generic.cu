// ring_generic.cu — the ring kernels for ANY power-of-two degree 32 <= d <= 1024 and any NTT-friendly prime
// q < 2^31 (SURVEY.md 8(f)4; the reference's own container tests run on (d, q) = (32, 193),
// tests/test_one_time_keys.py:12-33, and north_star asks for "d up to 1024").
//
// The shipped parameter sets (d = 256, q < 2^16) keep the register-resident half-warp kernels of ring.cu; every
// other (d, q) takes this path.  Work mapping, as north_star sketches it: ONE polynomial (vector) per WARP, the
// polynomial held in shared memory (4 bytes x d <= 4 KB), butterflies strided over the lanes with a __syncwarp per
// stage, 32-bit Shoup multiplication by the twiddles (valid for q < 2^31) and a 64-bit Barrett product for
// value x value multiplications.  Values are kept fully reduced in [0, q) between stages - this path trades the
// lazy-reduction tricks of ring.cu for one code path over every (d, q).
//
// Same entry points, formats and slot order as ring.cu: NTT slot p holds a(psi^(2 * bitrev_logd(p) + 1)), psi the
// least primitive 2d-th root of unity (the reference's `rou`).  Element types are template parameters:
// <int16_t, uint16_t> for q < 2^16 (the formats of include/lcb200.h), <int32_t, uint32_t> for wider moduli.
#include "engine.h"

namespace lcb {

namespace {

constexpr int GW = 4;              // warps (work items in flight) per block
constexpr int GBS = 32 * GW;

__device__ __forceinline__ uint32_t g_csub(uint32_t v, uint32_t q) { return v >= q ? v - q : v; }

// a any 32-bit value, w < q, ws = floor(w * 2^32 / q)  ->  a * w mod q in [0, q)      (q < 2^31)
__device__ __forceinline__ uint32_t g_shoup(uint32_t a, uint32_t w, uint32_t ws, uint32_t q) {
    return g_csub(a * w - __umulhi(a, ws) * q, q);
}

// a, b < q -> a * b mod q: 64-bit Barrett with mu = floor(2^64 / q) (quotient estimate short by at most 1)
__device__ __forceinline__ uint32_t g_mul(uint32_t a, uint32_t b, const GenRing& r) {
    const uint64_t p = (uint64_t)a * b;
    const uint64_t t = p - __umul64hi(p, r.mu64) * r.q;
    return g_csub(g_csub((uint32_t)t, r.q), r.q);
}

// signed coefficient of ANY magnitude its type allows -> residue in [0, q)
__device__ __forceinline__ uint32_t g_residue(int64_t v, const GenRing& r) {
    const uint64_t x = (uint64_t)(v + (int64_t)r.pos_off);      // pos_off = multiple of q >= 2^31: x >= 0
    const uint64_t t = x - __umul64hi(x, r.mu64) * r.q;
    return g_csub(g_csub((uint32_t)t, r.q), r.q);
}

__device__ __forceinline__ int32_t g_centre(uint32_t v, const GenRing& r) {
    return v > r.half ? (int32_t)v - (int32_t)r.q : (int32_t)v;
}

// Forward negacyclic NTT (Cooley-Tukey, natural order in, bit-reversed out) of x[0..d) in shared memory, values in
// [0, q) in and out.  Stage with half-length len has d/(2 len) groups; group g uses zeta index groups + g.
__device__ __forceinline__ void g_ntt_fwd(uint32_t* x, const GenRing& r, int lane) {
    int groups = 1, sh = r.logd - 1;
    for (int len = r.d >> 1; len >= 1; len >>= 1, groups <<= 1, --sh) {
        for (int b = lane; b < (r.d >> 1); b += 32) {
            const int g = b >> sh, j = b & (len - 1);
            const int i0 = ((2 * g) << sh) + j;
            const uint32_t t = g_shoup(x[i0 + len], __ldg(r.w + groups + g), __ldg(r.ws + groups + g), r.q);
            const uint32_t u = x[i0];
            x[i0] = g_csub(u + t, r.q);
            x[i0 + len] = g_csub(u + r.q - t, r.q);
        }
        __syncwarp();
    }
}

// Inverse (Gentleman-Sande, bit-reversed in, natural order out), scaled by d^-1.
__device__ __forceinline__ void g_ntt_inv(uint32_t* x, const GenRing& r, int lane) {
    int groups = r.d >> 1, sh = 0;
    for (int len = 1; len < r.d; len <<= 1, groups >>= 1, ++sh) {
        for (int b = lane; b < (r.d >> 1); b += 32) {
            const int g = b >> sh, j = b & (len - 1);
            const int i0 = ((2 * g) << sh) + j;
            const uint32_t u = x[i0], v = x[i0 + len];
            x[i0] = g_csub(u + v, r.q);
            x[i0 + len] = g_shoup(u + r.q - v, __ldg(r.iw + groups + g), __ldg(r.iws + groups + g), r.q);
        }
        __syncwarp();
    }
    for (int e = lane; e < r.d; e += 32) x[e] = g_shoup(x[e], r.dinv, r.dinv_s, r.q);
    __syncwarp();
}

struct WarpSlot {
    int lane, warp;
    uint32_t *x, *y, *z;      // three d-word arrays of this warp
};

__device__ __forceinline__ WarpSlot warp_slot(uint32_t* smem, int d) {
    WarpSlot s;
    s.lane = threadIdx.x & 31;
    s.warp = threadIdx.x >> 5;
    s.x = smem + (size_t)s.warp * 3 * d;
    s.y = s.x + d;
    s.z = s.y + d;
    return s;
}

// coefficient-form polynomial -> residues in x; returns this lane's (max |v|, #non-zero)
template <typename CT>
__device__ __forceinline__ void g_load_coef(uint32_t* x, const CT* __restrict__ p, const GenRing& r, int lane,
                                            int64_t& maxabs, int& nz) {
    for (int e = lane; e < r.d; e += 32) {
        const int64_t v = (int64_t)p[e];
        const int64_t av = v < 0 ? -v : v;
        maxabs = av > maxabs ? av : maxabs;
        nz += v != 0;
        x[e] = g_residue(v, r);
    }
    __syncwarp();
}

// sparse (index, coefficient) pairs in draw order -> dense residues in x
template <typename CT>
__device__ __forceinline__ void g_load_pairs(uint32_t* x, const CT* __restrict__ pairs, int wt, const GenRing& r, int lane) {
    for (int e = lane; e < r.d; e += 32) x[e] = 0;
    __syncwarp();
    for (int e = lane; e < wt; e += 32) {
        const int idx = (int)pairs[2 * e] & (r.d - 1);
        x[idx] = g_residue((int64_t)pairs[2 * e + 1], r);
    }
    __syncwarp();
}

template <typename CT>
__device__ __forceinline__ void g_store_coef(CT* __restrict__ p, const uint32_t* x, const GenRing& r, int lane) {
    for (int e = lane; e < r.d; e += 32) p[e] = (CT)g_centre(x[e], r);
}

__device__ __forceinline__ int warp_sum(int v) {
#pragma unroll
    for (int o = 16; o >= 1; o >>= 1) v += __shfl_xor_sync(0xFFFFFFFFu, v, o);
    return v;
}
__device__ __forceinline__ int64_t warp_max(int64_t v) {
#pragma unroll
    for (int o = 16; o >= 1; o >>= 1) {
        const int64_t w = __shfl_xor_sync(0xFFFFFFFFu, v, o);
        v = w > v ? w : v;
    }
    return v;
}

// ------------------------------------------------------------------------------------------------
template <typename CT, typename NT>
__global__ void __launch_bounds__(GBS) g_k_ntt_fwd(GenRing r, const CT* __restrict__ coef, int64_t npoly, NT* __restrict__ out) {
    extern __shared__ __align__(16) uint32_t smem[];
    const WarpSlot s = warp_slot(smem, r.d);
    for (int64_t it = (int64_t)blockIdx.x * GW + s.warp; it < npoly; it += (int64_t)gridDim.x * GW) {
        int64_t ma = 0;
        int nz = 0;
        g_load_coef(s.x, coef + it * r.d, r, s.lane, ma, nz);
        g_ntt_fwd(s.x, r, s.lane);
        for (int e = s.lane; e < r.d; e += 32) out[it * r.d + e] = (NT)s.x[e];
        __syncwarp();
    }
}

template <typename CT, typename NT>
__global__ void __launch_bounds__(GBS) g_k_ntt_inv(GenRing r, const NT* __restrict__ in, int64_t npoly, CT* __restrict__ coef) {
    extern __shared__ __align__(16) uint32_t smem[];
    const WarpSlot s = warp_slot(smem, r.d);
    for (int64_t it = (int64_t)blockIdx.x * GW + s.warp; it < npoly; it += (int64_t)gridDim.x * GW) {
        for (int e = s.lane; e < r.d; e += 32) s.x[e] = g_residue((int64_t)in[it * r.d + e], r);
        __syncwarp();
        g_ntt_inv(s.x, r, s.lane);
        g_store_coef(coef + it * r.d, s.x, r, s.lane);
        __syncwarp();
    }
}

template <typename CT>
__global__ void __launch_bounds__(GBS) g_k_poly_mul(GenRing r, const CT* __restrict__ a, const CT* __restrict__ b, int64_t npoly,
                                                    CT* __restrict__ out) {
    extern __shared__ __align__(16) uint32_t smem[];
    const WarpSlot s = warp_slot(smem, r.d);
    for (int64_t it = (int64_t)blockIdx.x * GW + s.warp; it < npoly; it += (int64_t)gridDim.x * GW) {
        int64_t ma = 0;
        int nz = 0;
        g_load_coef(s.x, a + it * r.d, r, s.lane, ma, nz);
        g_load_coef(s.y, b + it * r.d, r, s.lane, ma, nz);
        g_ntt_fwd(s.x, r, s.lane);
        g_ntt_fwd(s.y, r, s.lane);
        for (int e = s.lane; e < r.d; e += 32) s.x[e] = g_mul(s.x[e], s.y[e], r);
        __syncwarp();
        g_ntt_inv(s.x, r, s.lane);
        g_store_coef(out + it * r.d, s.x, r, s.lane);
        __syncwarp();
    }
}

// Polynomial.ntt_representation of lattice_algebra (parity level L3): rep[k] = a(rou^k), k in [0, 2d), centred.
template <typename CT>
__global__ void __launch_bounds__(GBS) g_k_ref_repr(GenRing r, const CT* __restrict__ coef, int64_t npoly, CT* __restrict__ out) {
    extern __shared__ __align__(16) uint32_t smem[];
    const WarpSlot s = warp_slot(smem, r.d);
    for (int64_t it = (int64_t)blockIdx.x * GW + s.warp; it < npoly; it += (int64_t)gridDim.x * GW) {
        int64_t ma = 0;
        int nz = 0;
        g_load_coef(s.x, coef + it * r.d, r, s.lane, ma, nz);
        // even exponents: the transform of the twisted polynomial c_j * psi^(-j)
        for (int e = s.lane; e < r.d; e += 32) s.y[e] = g_mul(s.x[e], __ldg(r.pw + ((2 * r.d - e) & (2 * r.d - 1))), r);
        __syncwarp();
        g_ntt_fwd(s.x, r, s.lane);
        g_ntt_fwd(s.y, r, s.lane);
        CT* o = out + it * 2 * r.d;
        for (int p = s.lane; p < r.d; p += 32) {
            const uint32_t i = __brev((uint32_t)p) >> (32 - r.logd);        // slot p -> exponent index
            o[2 * i + 1] = (CT)g_centre(s.x[p], r);
            o[2 * i] = (CT)g_centre(s.y[p], r);
        }
        __syncwarp();
    }
}

// y = key_ch * v for nvec coefficient-form vectors; optional NTT(v), NTT(y) and coefficient-form y outputs
template <typename CT, typename NT>
__global__ void __launch_bounds__(GBS) g_k_matvec(GenRing r, const uint32_t* __restrict__ a_hat, int l, const CT* __restrict__ vec_coef,
                                                  int64_t nvec, NT* __restrict__ vec_ntt, NT* __restrict__ y_ntt, CT* __restrict__ y_coef) {
    extern __shared__ __align__(16) uint32_t smem[];
    const WarpSlot s = warp_slot(smem, r.d);
    for (int64_t it = (int64_t)blockIdx.x * GW + s.warp; it < nvec; it += (int64_t)gridDim.x * GW) {
        for (int e = s.lane; e < r.d; e += 32) s.y[e] = 0;
        for (int i = 0; i < l; ++i) {
            int64_t ma = 0;
            int nz = 0;
            g_load_coef(s.x, vec_coef + (it * l + i) * r.d, r, s.lane, ma, nz);
            g_ntt_fwd(s.x, r, s.lane);
            for (int e = s.lane; e < r.d; e += 32) {
                if (vec_ntt) vec_ntt[(it * l + i) * r.d + e] = (NT)s.x[e];
                s.y[e] = g_csub(s.y[e] + g_mul(s.x[e], __ldg(a_hat + (size_t)i * r.d + e), r), r.q);
            }
            __syncwarp();
        }
        if (y_ntt)
            for (int e = s.lane; e < r.d; e += 32) y_ntt[it * r.d + e] = (NT)s.y[e];
        if (y_coef) {
            __syncwarp();
            g_ntt_inv(s.y, r, s.lane);
            g_store_coef(y_coef + it * r.d, s.y, r, s.lane);
        }
        __syncwarp();
    }
}

// sig = sk_left ** c + sk_right
template <typename CT, typename NT>
__global__ void __launch_bounds__(GBS) g_k_sign(GenRing r, int l, const NT* __restrict__ sk_ntt, const CT* __restrict__ ch_pairs, int ch_wt,
                                                int64_t n, CT* __restrict__ sig) {
    extern __shared__ __align__(16) uint32_t smem[];
    const WarpSlot s = warp_slot(smem, r.d);
    for (int64_t it = (int64_t)blockIdx.x * GW + s.warp; it < n; it += (int64_t)gridDim.x * GW) {
        g_load_pairs(s.z, ch_pairs + it * ch_wt * 2, ch_wt, r, s.lane);
        g_ntt_fwd(s.z, r, s.lane);
        for (int i = 0; i < l; ++i) {
            const NT* left = sk_ntt + (it * 2 * l + i) * r.d;
            const NT* right = left + (size_t)l * r.d;
            for (int e = s.lane; e < r.d; e += 32)
                s.x[e] = g_csub(g_mul(s.z[e], g_residue((int64_t)left[e], r), r) + g_residue((int64_t)right[e], r), r.q);
            __syncwarp();
            g_ntt_inv(s.x, r, s.lane);
            g_store_coef(sig + (it * l + i) * r.d, s.x, r, s.lane);
            __syncwarp();
        }
    }
}

// verdict = max|v| <= bd && max weight <= wt && key_ch * v == [vk_left * c] + rhs (+ extra)     (see ring.cu k_verify)
template <typename CT, typename NT>
__global__ void __launch_bounds__(GBS) g_k_verify(GenRing r, const uint32_t* __restrict__ a_hat, int l, const CT* __restrict__ vec_coef,
                                                  const NT* __restrict__ vk_ntt, const CT* __restrict__ ch_pairs, int ch_wt,
                                                  const NT* __restrict__ rhs_only, const NT* __restrict__ extra_rhs, int64_t n,
                                                  int64_t bd, int wt, uint8_t* __restrict__ verdict) {
    extern __shared__ __align__(16) uint32_t smem[];
    const WarpSlot s = warp_slot(smem, r.d);
    for (int64_t it = (int64_t)blockIdx.x * GW + s.warp; it < n; it += (int64_t)gridDim.x * GW) {
        for (int e = s.lane; e < r.d; e += 32) s.y[e] = 0;
        int64_t maxabs = 0;
        bool bad = false;
        for (int i = 0; i < l; ++i) {
            int nz = 0;
            g_load_coef(s.x, vec_coef + (it * l + i) * r.d, r, s.lane, maxabs, nz);
            bad |= warp_sum(nz) > wt;
            g_ntt_fwd(s.x, r, s.lane);
            for (int e = s.lane; e < r.d; e += 32)
                s.y[e] = g_csub(s.y[e] + g_mul(s.x[e], __ldg(a_hat + (size_t)i * r.d + e), r), r.q);
            __syncwarp();
        }
        bad |= warp_max(maxabs) > bd;
        bool eq = true;
        if (vk_ntt) {
            g_load_pairs(s.x, ch_pairs + it * ch_wt * 2, ch_wt, r, s.lane);
            g_ntt_fwd(s.x, r, s.lane);
        }
        for (int e = s.lane; e < r.d; e += 32) {
            uint32_t rhs;
            if (vk_ntt) {
                const uint32_t vl = g_residue((int64_t)vk_ntt[it * 2 * r.d + e], r);
                rhs = g_csub(g_mul(s.x[e], vl, r) + g_residue((int64_t)vk_ntt[it * 2 * r.d + r.d + e], r), r.q);
            } else {
                rhs = g_residue((int64_t)rhs_only[it * r.d + e], r);
            }
            if (extra_rhs) rhs = g_csub(rhs + g_residue((int64_t)extra_rhs[it * r.d + e], r), r.q);
            eq &= s.y[e] == rhs;
        }
        const unsigned votes = __ballot_sync(0xFFFFFFFFu, eq && !bad);
        if (s.lane == 0) verdict[it] = votes == 0xFFFFFFFFu ? 1 : 0;
        __syncwarp();
    }
}

template <typename CT>
__global__ void g_k_vec_addsub(GenRing r, const CT* __restrict__ a, const CT* __restrict__ b, int64_t nelem, int sub, CT* __restrict__ out) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nelem; i += (int64_t)gridDim.x * blockDim.x) {
        // each operand reduced on its own: a +- b of two int32 values can reach -2^32, below what pos_off lifts
        const uint32_t x = g_residue((int64_t)a[i], r), y = g_residue((int64_t)b[i], r);
        out[i] = (CT)g_centre(g_csub(sub ? x + r.q - y : x + y, r.q), r);
    }
}

// BKLM aggregate, monomial coefficients (ring.cu k_agg_partial); partial holds residues (int32) or, for q >= 2^16,
// 64-bit sums (PT = int64_t)
template <typename CT, typename PT>
__global__ void __launch_bounds__(GBS) g_k_agg_partial(GenRing r, int l, const CT* __restrict__ sigs, const CT* __restrict__ ag_pairs,
                                                       int64_t count, PT* __restrict__ partial) {
    extern __shared__ __align__(16) uint32_t smem[];
    const WarpSlot s = warp_slot(smem, r.d);
    const int poly = blockIdx.y;
    for (int e = s.lane; e < r.d; e += 32) s.y[e] = 0;
    __syncwarp();
    for (int64_t t = (int64_t)blockIdx.x * GW + s.warp; t < count; t += (int64_t)gridDim.x * GW) {
        const int k = (int)ag_pairs[2 * t] & (r.d - 1);
        const int64_t sg = (int64_t)ag_pairs[2 * t + 1];
        const CT* row = sigs + (t * l + poly) * r.d;
        for (int p = s.lane; p < r.d; p += 32) {
            int64_t v = (int64_t)row[(p - k) & (r.d - 1)] * sg;
            v = p < k ? -v : v;
            s.y[p] = g_csub(s.y[p] + g_residue(v, r), r.q);
        }
    }
    __syncwarp();
    for (int e = s.lane; e < r.d; e += 32) atomicAdd(&partial[poly * r.d + e], (PT)s.y[e]);
}

// BKLM aggregate_verify right-hand side (ring.cu k_aggv_partial)
template <typename CT, typename NT, typename PT>
__global__ void __launch_bounds__(GBS) g_k_aggv_partial(GenRing r, const NT* __restrict__ vk_ntt, const CT* __restrict__ ch_pairs, int ch_wt,
                                                        const CT* __restrict__ ag_pairs, int64_t count, PT* __restrict__ partial) {
    extern __shared__ __align__(16) uint32_t smem[];
    const WarpSlot s = warp_slot(smem, r.d);
    for (int e = s.lane; e < r.d; e += 32) s.y[e] = 0;
    __syncwarp();
    for (int64_t it = (int64_t)blockIdx.x * GW + s.warp; it < count; it += (int64_t)gridDim.x * GW) {
        g_load_pairs(s.x, ch_pairs + it * ch_wt * 2, ch_wt, r, s.lane);
        g_ntt_fwd(s.x, r, s.lane);
        const uint32_t kk = (uint32_t)ag_pairs[2 * it] & (uint32_t)(r.d - 1);
        const bool neg = (int64_t)ag_pairs[2 * it + 1] < 0;
        for (int e = s.lane; e < r.d; e += 32) {
            const uint32_t vl = g_residue((int64_t)vk_ntt[it * 2 * r.d + e], r);
            const uint32_t vr = g_residue((int64_t)vk_ntt[it * 2 * r.d + r.d + e], r);
            const uint32_t t = g_csub(g_mul(s.x[e], vl, r) + vr, r.q);
            const uint32_t odd = 2 * (__brev((uint32_t)e) >> (32 - r.logd)) + 1;
            uint32_t u = g_mul(t, __ldg(r.pw + ((odd * kk) & (uint32_t)(2 * r.d - 1))), r);
            u = neg ? g_csub(r.q - u, r.q) : u;
            s.y[e] = g_csub(s.y[e] + u, r.q);
        }
        __syncwarp();
    }
    for (int e = s.lane; e < r.d; e += 32) atomicAdd(&partial[e], (PT)s.y[e]);
}

// ---- general aggregation coefficients (ag_wt > 1 or ag_bd > 1; bklm_one_time_agg_sigs.py:15-19 leaves both as editable
// tables and computes sig ** ag_coef / (...) * ag_coef with full polynomial products, :96,114-115).  Coefficient i is a
// sparse polynomial given as ag_wt (index, value) pairs.
// aggregate: per signature NTT(ag_i) and l forward transforms, products accumulated in the NTT domain in a per-block
// shared array [l][d]; each block inverse-transforms its sum once and adds it to partial, which therefore stays a
// coefficient-domain sum like the monomial kernel's.  One launch covers the polynomials p0 .. p0 + np - 1 of the vector
// (the accumulator of all l may exceed the shared memory of a block; see g_launch_agg_partial_poly).
template <typename CT, typename PT>
__global__ void __launch_bounds__(GBS) g_k_agg_partial_poly(GenRing r, int l, int p0, int np, const CT* __restrict__ sigs,
                                                            const CT* __restrict__ ag_pairs, int ag_wt, int64_t count,
                                                            PT* __restrict__ partial) {
    extern __shared__ __align__(16) uint32_t smem[];
    const WarpSlot s = warp_slot(smem, r.d);
    uint32_t* acc = smem + (size_t)GW * 3 * r.d;               // [np][d], shared by the block
    for (int e = threadIdx.x; e < np * r.d; e += GBS) acc[e] = 0;
    __syncthreads();
    for (int64_t t = (int64_t)blockIdx.x * GW + s.warp; t < count; t += (int64_t)gridDim.x * GW) {
        g_load_pairs(s.z, ag_pairs + t * ag_wt * 2, ag_wt, r, s.lane);
        g_ntt_fwd(s.z, r, s.lane);
        for (int i = 0; i < np; ++i) {
            int64_t ma = 0;
            int nz = 0;
            g_load_coef(s.x, sigs + (t * l + p0 + i) * r.d, r, s.lane, ma, nz);
            g_ntt_fwd(s.x, r, s.lane);
            for (int e = s.lane; e < r.d; e += 32) {
                const uint32_t v = g_mul(s.x[e], s.z[e], r);
                // modular add on a word other warps add to as well: compare-and-swap loop
                uint32_t* a = acc + (size_t)i * r.d + e;
                uint32_t old = *a, assumed;
                do {
                    assumed = old;
                    old = atomicCAS(a, assumed, g_csub(assumed + v, r.q));
                } while (old != assumed);
            }
            __syncwarp();
        }
    }
    __syncthreads();
    for (int i = s.warp; i < np; i += GW) {
        g_ntt_inv(acc + (size_t)i * r.d, r, s.lane);
        for (int e = s.lane; e < r.d; e += 32) atomicAdd(&partial[(size_t)(p0 + i) * r.d + e], (PT)acc[(size_t)i * r.d + e]);
    }
}

template <typename CT, typename NT, typename PT>
__global__ void __launch_bounds__(GBS) g_k_aggv_partial_poly(GenRing r, const NT* __restrict__ vk_ntt, const CT* __restrict__ ch_pairs,
                                                             int ch_wt, const CT* __restrict__ ag_pairs, int ag_wt, int64_t count,
                                                             PT* __restrict__ partial) {
    extern __shared__ __align__(16) uint32_t smem[];
    const WarpSlot s = warp_slot(smem, r.d);
    for (int e = s.lane; e < r.d; e += 32) s.y[e] = 0;
    __syncwarp();
    for (int64_t it = (int64_t)blockIdx.x * GW + s.warp; it < count; it += (int64_t)gridDim.x * GW) {
        g_load_pairs(s.x, ch_pairs + it * ch_wt * 2, ch_wt, r, s.lane);
        g_ntt_fwd(s.x, r, s.lane);
        g_load_pairs(s.z, ag_pairs + it * ag_wt * 2, ag_wt, r, s.lane);
        g_ntt_fwd(s.z, r, s.lane);
        for (int e = s.lane; e < r.d; e += 32) {
            const uint32_t vl = g_residue((int64_t)vk_ntt[it * 2 * r.d + e], r);
            const uint32_t vr = g_residue((int64_t)vk_ntt[it * 2 * r.d + r.d + e], r);
            const uint32_t t = g_csub(g_mul(s.x[e], vl, r) + vr, r.q);
            s.y[e] = g_csub(s.y[e] + g_mul(t, s.z[e], r), r.q);
        }
        __syncwarp();
    }
    for (int e = s.lane; e < r.d; e += 32) atomicAdd(&partial[e], (PT)s.y[e]);
}

template <typename CT, typename PT>
__global__ void g_k_agg_finish(GenRing r, const PT* __restrict__ partial, int n, CT* __restrict__ out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    out[i] = (CT)g_centre(g_residue((int64_t)partial[i], r), r);
}

// bounds on ag_sig (with lower limits), key_ch * ag_sig == partial sum; one warp
template <typename CT, typename PT>
__global__ void __launch_bounds__(32) g_k_aggv_finish(GenRing r, const uint32_t* __restrict__ a_hat, int l, const PT* __restrict__ partial,
                                                      const CT* __restrict__ ag_sig, int64_t total, int64_t ag_cap, int64_t avf_bd,
                                                      int avf_wt, uint8_t* __restrict__ verdict) {
    extern __shared__ __align__(16) uint32_t smem[];
    const WarpSlot s = warp_slot(smem, r.d);
    for (int e = s.lane; e < r.d; e += 32) s.y[e] = 0;
    int64_t maxabs = 0;
    int maxw = 0;
    for (int i = 0; i < l; ++i) {
        int nz = 0;
        g_load_coef(s.x, ag_sig + (size_t)i * r.d, r, s.lane, maxabs, nz);
        nz = warp_sum(nz);
        maxw = nz > maxw ? nz : maxw;
        g_ntt_fwd(s.x, r, s.lane);
        for (int e = s.lane; e < r.d; e += 32)
            s.y[e] = g_csub(s.y[e] + g_mul(s.x[e], __ldg(a_hat + (size_t)i * r.d + e), r), r.q);
        __syncwarp();
    }
    maxabs = warp_max(maxabs);
    bool ok = maxabs >= 1 && maxabs <= avf_bd && maxw >= 1 && maxw <= avf_wt && total >= 1 && total <= ag_cap;
    for (int e = s.lane; e < r.d; e += 32) ok &= s.y[e] == g_residue((int64_t)partial[e], r);
    const unsigned votes = __ballot_sync(0xFFFFFFFFu, ok);
    if (s.lane == 0) verdict[0] = votes == 0xFFFFFFFFu ? 1 : 0;
}

inline size_t g_smem(const GenRing& r, int warps = GW) { return (size_t)warps * 3 * r.d * sizeof(uint32_t); }

inline unsigned g_grid(int64_t items, int num_sms) {
    int64_t need = (items + GW - 1) / GW;
    int64_t cap = (int64_t)num_sms * 8;
    return (unsigned)(need < cap ? (need < 1 ? 1 : need) : cap);
}

}  // namespace

// ---- host launchers: the generic twins of ring.cu's, selected by api.cu when ctx->generic ----------------------
#define G_LAUNCH(kernel, grid, block, smem, st, ...)                                                   \
    do {                                                                                               \
        cudaError_t e_ = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(smem)); \
        if (e_ != cudaSuccess) return e_;                                                              \
        kernel<<<grid, block, smem, st>>>(__VA_ARGS__);                                                \
        return cudaGetLastError();                                                                     \
    } while (0)

cudaError_t g_launch_ntt_fwd(const GenCtx& c, const void* coef, int64_t npoly, void* out, cudaStream_t st) {
    if (npoly <= 0) return cudaSuccess;
    if (c.wide) G_LAUNCH((g_k_ntt_fwd<int32_t, uint32_t>), g_grid(npoly, c.num_sms), GBS, g_smem(c.r), st, c.r, (const int32_t*)coef, npoly, (uint32_t*)out);
    G_LAUNCH((g_k_ntt_fwd<int16_t, uint16_t>), g_grid(npoly, c.num_sms), GBS, g_smem(c.r), st, c.r, (const int16_t*)coef, npoly, (uint16_t*)out);
}

cudaError_t g_launch_ntt_inv(const GenCtx& c, const void* in, int64_t npoly, void* coef, cudaStream_t st) {
    if (npoly <= 0) return cudaSuccess;
    if (c.wide) G_LAUNCH((g_k_ntt_inv<int32_t, uint32_t>), g_grid(npoly, c.num_sms), GBS, g_smem(c.r), st, c.r, (const uint32_t*)in, npoly, (int32_t*)coef);
    G_LAUNCH((g_k_ntt_inv<int16_t, uint16_t>), g_grid(npoly, c.num_sms), GBS, g_smem(c.r), st, c.r, (const uint16_t*)in, npoly, (int16_t*)coef);
}

cudaError_t g_launch_poly_mul(const GenCtx& c, const void* a, const void* b, int64_t npoly, void* out, cudaStream_t st) {
    if (npoly <= 0) return cudaSuccess;
    if (c.wide) G_LAUNCH((g_k_poly_mul<int32_t>), g_grid(npoly, c.num_sms), GBS, g_smem(c.r), st, c.r, (const int32_t*)a, (const int32_t*)b, npoly, (int32_t*)out);
    G_LAUNCH((g_k_poly_mul<int16_t>), g_grid(npoly, c.num_sms), GBS, g_smem(c.r), st, c.r, (const int16_t*)a, (const int16_t*)b, npoly, (int16_t*)out);
}

cudaError_t g_launch_ref_repr(const GenCtx& c, const void* coef, int64_t npoly, void* out, cudaStream_t st) {
    if (npoly <= 0) return cudaSuccess;
    if (c.wide) G_LAUNCH((g_k_ref_repr<int32_t>), g_grid(npoly, c.num_sms), GBS, g_smem(c.r), st, c.r, (const int32_t*)coef, npoly, (int32_t*)out);
    G_LAUNCH((g_k_ref_repr<int16_t>), g_grid(npoly, c.num_sms), GBS, g_smem(c.r), st, c.r, (const int16_t*)coef, npoly, (int16_t*)out);
}

cudaError_t g_launch_matvec(const GenCtx& c, const void* vec_coef, int64_t nvec, void* vec_ntt, void* y_ntt, void* y_coef,
                            cudaStream_t st) {
    if (nvec <= 0) return cudaSuccess;
    if (c.wide) G_LAUNCH((g_k_matvec<int32_t, uint32_t>), g_grid(nvec, c.num_sms), GBS, g_smem(c.r), st, c.r, c.a_hat, c.l, (const int32_t*)vec_coef, nvec, (uint32_t*)vec_ntt, (uint32_t*)y_ntt, (int32_t*)y_coef);
    G_LAUNCH((g_k_matvec<int16_t, uint16_t>), g_grid(nvec, c.num_sms), GBS, g_smem(c.r), st, c.r, c.a_hat, c.l, (const int16_t*)vec_coef, nvec, (uint16_t*)vec_ntt, (uint16_t*)y_ntt, (int16_t*)y_coef);
}

cudaError_t g_launch_sign(const GenCtx& c, const void* sk_ntt, const void* ch_pairs, int ch_wt, int64_t n, void* sig, cudaStream_t st) {
    if (n <= 0) return cudaSuccess;
    if (c.wide) G_LAUNCH((g_k_sign<int32_t, uint32_t>), g_grid(n, c.num_sms), GBS, g_smem(c.r), st, c.r, c.l, (const uint32_t*)sk_ntt, (const int32_t*)ch_pairs, ch_wt, n, (int32_t*)sig);
    G_LAUNCH((g_k_sign<int16_t, uint16_t>), g_grid(n, c.num_sms), GBS, g_smem(c.r), st, c.r, c.l, (const uint16_t*)sk_ntt, (const int16_t*)ch_pairs, ch_wt, n, (int16_t*)sig);
}

cudaError_t g_launch_verify(const GenCtx& c, const void* vec_coef, const void* vk_ntt, const void* ch_pairs, int ch_wt,
                            const void* rhs_only, const void* extra_rhs, int64_t n, int64_t bd, int wt, uint8_t* verdict,
                            cudaStream_t st) {
    if (n <= 0) return cudaSuccess;
    if (c.wide) G_LAUNCH((g_k_verify<int32_t, uint32_t>), g_grid(n, c.num_sms), GBS, g_smem(c.r), st, c.r, c.a_hat, c.l, (const int32_t*)vec_coef, (const uint32_t*)vk_ntt, (const int32_t*)ch_pairs, ch_wt, (const uint32_t*)rhs_only, (const uint32_t*)extra_rhs, n, bd, wt, verdict);
    G_LAUNCH((g_k_verify<int16_t, uint16_t>), g_grid(n, c.num_sms), GBS, g_smem(c.r), st, c.r, c.a_hat, c.l, (const int16_t*)vec_coef, (const uint16_t*)vk_ntt, (const int16_t*)ch_pairs, ch_wt, (const uint16_t*)rhs_only, (const uint16_t*)extra_rhs, n, bd, wt, verdict);
}

cudaError_t g_launch_vec_addsub(const GenCtx& c, const void* a, const void* b, int64_t nelem, int sub, void* out, cudaStream_t st) {
    if (nelem <= 0) return cudaSuccess;
    int64_t need = (nelem + 255) / 256, cap = (int64_t)c.num_sms * 8;
    const unsigned grid = (unsigned)(need < cap ? need : cap);
    if (c.wide) { g_k_vec_addsub<int32_t><<<grid, 256, 0, st>>>(c.r, (const int32_t*)a, (const int32_t*)b, nelem, sub, (int32_t*)out); return cudaGetLastError(); }
    g_k_vec_addsub<int16_t><<<grid, 256, 0, st>>>(c.r, (const int16_t*)a, (const int16_t*)b, nelem, sub, (int16_t*)out);
    return cudaGetLastError();
}

cudaError_t g_launch_agg_partial(const GenCtx& c, const void* sigs, const void* ag_pairs, int64_t count, void* partial, cudaStream_t st) {
    if (count <= 0) return cudaSuccess;
    int64_t need = (count + 8 * GW - 1) / (8 * GW), cap = (int64_t)c.num_sms * 8 / c.l + 1;
    dim3 grid((unsigned)(need < cap ? need : cap), (unsigned)c.l);
    if (c.wide) G_LAUNCH((g_k_agg_partial<int32_t, unsigned long long>), grid, GBS, g_smem(c.r), st, c.r, c.l, (const int32_t*)sigs, (const int32_t*)ag_pairs, count, (unsigned long long*)partial);
    G_LAUNCH((g_k_agg_partial<int16_t, int32_t>), grid, GBS, g_smem(c.r), st, c.r, c.l, (const int16_t*)sigs, (const int16_t*)ag_pairs, count, (int32_t*)partial);
}

// The block's [np][d] accumulator sits beside the warps' work arrays.  At d = 1024 a whole vector of l >= 45 polynomials
// exceeds the opt-in shared-memory limit (227 KB on the B200; l = 64 would need 304 KB), so the vector is summed in slices
// of as many polynomials as fit, one launch each.
template <typename CT, typename PT>
cudaError_t g_agg_partial_poly_slices(const GenCtx& c, const CT* sigs, const CT* ag_pairs, int ag_wt, int64_t count, PT* partial,
                                      cudaStream_t st) {
    const size_t row = (size_t)c.r.d * sizeof(uint32_t);
    const int fit = c.smem_optin > g_smem(c.r) ? (int)((c.smem_optin - g_smem(c.r)) / row) : 0;
    const int slice = fit < c.l ? fit : c.l;
    if (slice < 1) return cudaErrorInvalidConfiguration;
    cudaError_t e = cudaFuncSetAttribute(g_k_agg_partial_poly<CT, PT>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         (int)(g_smem(c.r) + slice * row));
    if (e != cudaSuccess) return e;
    const unsigned grid = g_grid(count, c.num_sms / 2 + 1);
    for (int p0 = 0; p0 < c.l; p0 += slice) {
        const int np = c.l - p0 < slice ? c.l - p0 : slice;
        g_k_agg_partial_poly<CT, PT><<<grid, GBS, g_smem(c.r) + np * row, st>>>(c.r, c.l, p0, np, sigs, ag_pairs, ag_wt, count, partial);
        if ((e = cudaGetLastError()) != cudaSuccess) return e;
    }
    return cudaSuccess;
}

cudaError_t g_launch_agg_partial_poly(const GenCtx& c, const void* sigs, const void* ag_pairs, int ag_wt, int64_t count,
                                      void* partial, cudaStream_t st) {
    if (count <= 0) return cudaSuccess;
    if (c.wide)
        return g_agg_partial_poly_slices(c, (const int32_t*)sigs, (const int32_t*)ag_pairs, ag_wt, count, (unsigned long long*)partial, st);
    return g_agg_partial_poly_slices(c, (const int16_t*)sigs, (const int16_t*)ag_pairs, ag_wt, count, (int32_t*)partial, st);
}

cudaError_t g_launch_aggv_partial_poly(const GenCtx& c, const void* vk_ntt, const void* ch_pairs, int ch_wt, const void* ag_pairs,
                                       int ag_wt, int64_t count, void* partial, cudaStream_t st) {
    if (count <= 0) return cudaSuccess;
    const unsigned grid = g_grid(count, c.num_sms);
    if (c.wide) G_LAUNCH((g_k_aggv_partial_poly<int32_t, uint32_t, unsigned long long>), grid, GBS, g_smem(c.r), st, c.r, (const uint32_t*)vk_ntt, (const int32_t*)ch_pairs, ch_wt, (const int32_t*)ag_pairs, ag_wt, count, (unsigned long long*)partial);
    G_LAUNCH((g_k_aggv_partial_poly<int16_t, uint16_t, int32_t>), grid, GBS, g_smem(c.r), st, c.r, (const uint16_t*)vk_ntt, (const int16_t*)ch_pairs, ch_wt, (const int16_t*)ag_pairs, ag_wt, count, (int32_t*)partial);
}

cudaError_t g_launch_agg_finish(const GenCtx& c, const void* partial, void* ag_sig, cudaStream_t st) {
    const int n = c.l * c.r.d;
    if (c.wide) { g_k_agg_finish<int32_t, unsigned long long><<<(n + 255) / 256, 256, 0, st>>>(c.r, (const unsigned long long*)partial, n, (int32_t*)ag_sig); return cudaGetLastError(); }
    g_k_agg_finish<int16_t, int32_t><<<(n + 255) / 256, 256, 0, st>>>(c.r, (const int32_t*)partial, n, (int16_t*)ag_sig);
    return cudaGetLastError();
}

cudaError_t g_launch_aggv_partial(const GenCtx& c, const void* vk_ntt, const void* ch_pairs, int ch_wt, const void* ag_pairs,
                                  int64_t count, void* partial, cudaStream_t st) {
    if (count <= 0) return cudaSuccess;
    const unsigned grid = g_grid(count, c.num_sms);
    if (c.wide) G_LAUNCH((g_k_aggv_partial<int32_t, uint32_t, unsigned long long>), grid, GBS, g_smem(c.r), st, c.r, (const uint32_t*)vk_ntt, (const int32_t*)ch_pairs, ch_wt, (const int32_t*)ag_pairs, count, (unsigned long long*)partial);
    G_LAUNCH((g_k_aggv_partial<int16_t, uint16_t, int32_t>), grid, GBS, g_smem(c.r), st, c.r, (const uint16_t*)vk_ntt, (const int16_t*)ch_pairs, ch_wt, (const int16_t*)ag_pairs, count, (int32_t*)partial);
}

cudaError_t g_launch_aggv_finish(const GenCtx& c, const void* partial, const void* ag_sig, int64_t total, int64_t ag_cap,
                                 int64_t avf_bd, int avf_wt, uint8_t* verdict, cudaStream_t st) {
    if (c.wide) G_LAUNCH((g_k_aggv_finish<int32_t, unsigned long long>), 1, 32, g_smem(c.r, 1), st, c.r, c.a_hat, c.l, (const unsigned long long*)partial, (const int32_t*)ag_sig, total, ag_cap, avf_bd, avf_wt, verdict);
    G_LAUNCH((g_k_aggv_finish<int16_t, int32_t>), 1, 32, g_smem(c.r, 1), st, c.r, c.a_hat, c.l, (const int32_t*)partial, (const int16_t*)ag_sig, total, ag_cap, avf_bd, avf_wt, verdict);
}

}  // namespace lcb
