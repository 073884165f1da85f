// wire.cu — packed wire format for keys and signatures (SURVEY 8(f)2; sm_100a).
//
// The reference has no serialisation at all: keys print as memory addresses and signatures are Python
// objects (one_time_keys.py:197-237).  This is the engine's own, opt-in format: every polynomial is its
// 256 values v_i = (x_i + bias) mod 2^16, each stored in `bits` bits, value i at bit offset i*bits,
// least significant bit first (byte = offset >> 3, bit = offset & 7) - 32*bits bytes per polynomial.
//   signatures : x = centred coefficient, bias = vf_bd, bits = ceil(log2(2*vf_bd + 1))   (11 / 13)
//   NTT-form keys : x = slot value in [0, q), bias = 0, bits = ceil(log2 q)               (14 / 16)
//   adaptor witnesses : x = centred coefficient, bias = wit_bd, bits = ceil(log2(2*wit_bd + 1))   (2)
// All kernels are pure HBM streams: one warp per polynomial, global traffic as 16-byte / 4-byte
// coalesced accesses, the bit shuffling in a per-warp shared-memory row.
#include "engine.h"

namespace lcb {

namespace {

constexpr int WBS = 256;                       // threads per block
constexpr int WARPS = WBS / 32;
constexpr int ROW_WORDS = 8 * 16 + 4;          // packed polynomial at 16 bits + slack read by the funnel

__global__ void __launch_bounds__(WBS) k_pack(const uint16_t* __restrict__ in, int64_t npoly, int bits, uint32_t bias,
                                              uint32_t* __restrict__ out, uint8_t* __restrict__ in_range) {
    __shared__ uint32_t rows[WARPS][ROW_WORDS];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    uint32_t* row = rows[warp];
    uint8_t* rowb = reinterpret_cast<uint8_t*>(row);
    const uint32_t limit = 1u << bits;
    const int words = 8 * bits;
    for (int64_t p = (int64_t)blockIdx.x * WARPS + warp; p < npoly; p += (int64_t)gridDim.x * WARPS) {
        const uint4 raw = __ldg(reinterpret_cast<const uint4*>(in + p * D) + lane);     // 8 values of this lane
        const uint32_t w[4] = {raw.x, raw.y, raw.z, raw.w};
        // 8 values x bits = `bits` whole bytes per lane, at byte lane*bits of the row
        uint64_t acc = 0;
        int fill = 0, nb = 0;
        bool ok = true;
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const uint32_t v = (((w[i >> 1] >> (16 * (i & 1))) & 0xFFFFu) + bias) & 0xFFFFu;
            ok = ok && v < limit;
            acc |= (uint64_t)(v & (limit - 1)) << fill;
            fill += bits;
            while (fill >= 8) {
                rowb[lane * bits + nb++] = (uint8_t)acc;
                acc >>= 8;
                fill -= 8;
            }
        }
        ok = __all_sync(0xFFFFFFFFu, ok);
        __syncwarp();
        uint32_t* o = out + p * words;
        for (int k = lane; k < words; k += 32) o[k] = row[k];
        if (in_range && lane == 0) in_range[p] = ok ? 1 : 0;
        __syncwarp();
    }
}

// The 8 values of a lane (value 8 lane + i of the polynomial, already biased, < 2^16) as `bits` whole bytes at byte
// lane*bits of the warp's row; false if one of them needs more than `bits` bits
__device__ __forceinline__ bool pack_lane(uint8_t* rowb, int lane, int bits, const uint32_t (&v)[8]) {
    const uint32_t limit = 1u << bits;
    uint64_t acc = 0;
    int fill = 0, nb = 0;
    bool ok = true;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        ok = ok && v[i] < limit;
        acc |= (uint64_t)(v[i] & (limit - 1)) << fill;
        fill += bits;
        while (fill >= 8) {
            rowb[lane * bits + nb++] = (uint8_t)acc;
            acc >>= 8;
            fill -= 8;
        }
    }
    return ok;
}

// BKLM aggregates straight into the wire format: k_agg_finish followed by k_pack, without the int16 aggregates making a
// round trip through HBM.  partial int32[npoly][256] (|x| < 2^30) -> x mod q by Barrett reduction of x + off (off: a
// multiple of q >= 2^30) -> centred -> (x + bias) mod 2^16 in `bits` bits, in_range[p] as k_pack sets it.
__global__ void __launch_bounds__(WBS) k_agg_finish_pack(ModQ m, uint32_t off, const int32_t* __restrict__ partial,
                                                         int64_t npoly, int bits, uint32_t bias, uint32_t* __restrict__ out,
                                                         uint8_t* __restrict__ in_range) {
    __shared__ uint32_t rows[WARPS][ROW_WORDS];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    uint32_t* row = rows[warp];
    uint8_t* rowb = reinterpret_cast<uint8_t*>(row);
    const int words = 8 * bits;
    for (int64_t p = (int64_t)blockIdx.x * WARPS + warp; p < npoly; p += (int64_t)gridDim.x * WARPS) {
        const int4* src = reinterpret_cast<const int4*>(partial + p * D) + 2 * lane;
        const int4 a = __ldg(src), b = __ldg(src + 1);
        const int x[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
        uint32_t v[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) v[i] = ((uint32_t)center(barrett_full((uint32_t)x[i] + off, m), m) + bias) & 0xFFFFu;
        bool ok = pack_lane(rowb, lane, bits, v);
        ok = __all_sync(0xFFFFFFFFu, ok);
        __syncwarp();
        uint32_t* o = out + p * words;
        for (int k = lane; k < words; k += 32) o[k] = row[k];
        if (in_range && lane == 0) in_range[p] = ok ? 1 : 0;
        __syncwarp();
    }
}

__global__ void __launch_bounds__(WBS) k_unpack(const uint32_t* __restrict__ in, int64_t npoly, int bits, uint32_t bias,
                                                uint16_t* __restrict__ out) {
    __shared__ uint32_t rows[WARPS][ROW_WORDS];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    uint32_t* row = rows[warp];
    const uint32_t mask = (1u << bits) - 1;
    const int words = 8 * bits;
    for (int k = lane; k < ROW_WORDS; k += 32) row[k] = 0;
    for (int64_t p = (int64_t)blockIdx.x * WARPS + warp; p < npoly; p += (int64_t)gridDim.x * WARPS) {
        __syncwarp();
        const uint32_t* src = in + p * words;
        for (int k = lane; k < words; k += 32) row[k] = __ldg(src + k);
        __syncwarp();
        uint32_t w[4];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const int pos = (lane * 8 + i) * bits;
            const uint32_t v = __funnelshift_r(row[pos >> 5], row[(pos >> 5) + 1], pos & 31) & mask;
            const uint32_t x = (v - bias) & 0xFFFFu;
            if (i & 1) w[i >> 1] |= x << 16;
            else w[i >> 1] = x;
        }
        reinterpret_cast<uint4*>(out + p * D)[lane] = make_uint4(w[0], w[1], w[2], w[3]);
    }
}

// The 8 values of a lane from a packed row staged in the warp's shared row, as k_unpack decodes them: (v - bias) mod 2^16
// read as int16
__device__ __forceinline__ void unpack_lane_s16(const uint32_t* row, int lane, int bits, uint32_t bias, int (&x)[8]) {
    const uint32_t mask = (1u << bits) - 1;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const int pos = (lane * 8 + i) * bits;
        const uint32_t v = __funnelshift_r(row[pos >> 5], row[(pos >> 5) + 1], pos & 31) & mask;
        x[i] = (int16_t)((v - bias) & 0xFFFFu);
    }
}

// Adaptor adapt / extract on the wire format in one pass: unpack both operands -> k_vec_addsub -> k_pack, without the
// int16 rows making a round trip through HBM.  out = a + b (sub = 0) or a - b (sub = 1), reduced and centred exactly as
// k_vec_addsub does, then (r + bias) mod 2^16 in `bits` bits and in_range[p] as k_pack sets it.  One warp per polynomial;
// every width is a run-time argument.
__global__ void __launch_bounds__(WBS) k_addsub_packed(ModQ m, const uint32_t* __restrict__ a, int a_bits, uint32_t a_bias,
                                                       const uint32_t* __restrict__ b, int b_bits, uint32_t b_bias, int sub,
                                                       int64_t npoly, int bits, uint32_t bias, uint32_t* __restrict__ out,
                                                       uint8_t* __restrict__ in_range) {
    __shared__ uint32_t rows[2][WARPS][ROW_WORDS];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    uint32_t* ra = rows[0][warp];
    uint32_t* rb = rows[1][warp];
    uint8_t* rowb = reinterpret_cast<uint8_t*>(ra);
    const int a_words = 8 * a_bits, b_words = 8 * b_bits, words = 8 * bits;
    const int two_cq_q = 2 * (int)m.cq + (int)m.q;
    for (int k = lane; k < ROW_WORDS; k += 32) ra[k] = rb[k] = 0;
    for (int64_t p = (int64_t)blockIdx.x * WARPS + warp; p < npoly; p += (int64_t)gridDim.x * WARPS) {
        __syncwarp();
        for (int k = lane; k < a_words; k += 32) ra[k] = __ldg(a + p * a_words + k);
        for (int k = lane; k < b_words; k += 32) rb[k] = __ldg(b + p * b_words + k);
        __syncwarp();
        int xa[8], xb[8];
        unpack_lane_s16(ra, lane, a_bits, a_bias, xa);
        unpack_lane_s16(rb, lane, b_bits, b_bias, xb);
        uint32_t v[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const int y = sub ? -xb[i] : xb[i];
            v[i] = ((uint32_t)center(barrett_full((uint32_t)(xa[i] + y + two_cq_q), m), m) + bias) & 0xFFFFu;
        }
        __syncwarp();                                   // every lane has decoded its values: the row takes the output
        bool ok = pack_lane(rowb, lane, bits, v);
        ok = __all_sync(0xFFFFFFFFu, ok);
        __syncwarp();
        uint32_t* o = out + p * words;
        for (int k = lane; k < words; k += 32) o[k] = ra[k];
        if (in_range && lane == 0) in_range[p] = ok ? 1 : 0;
    }
}

int wire_grid(int64_t npoly, int num_sms) {
    const int64_t blocks = (npoly + WARPS - 1) / WARPS;
    const int64_t cap = (int64_t)num_sms * 8;          // 8 resident 256-thread blocks per SM, grid-stride beyond
    return (int)(blocks < cap ? blocks : cap);
}

}  // namespace

cudaError_t launch_pack(const RingCtx& c, const void* in, int64_t npoly, int bits, int bias, uint8_t* out,
                        uint8_t* in_range, cudaStream_t st) {
    if (npoly <= 0) return cudaSuccess;
    if (bits < 1 || bits > 16) return cudaErrorInvalidValue;
    k_pack<<<wire_grid(npoly, c.num_sms), WBS, 0, st>>>(static_cast<const uint16_t*>(in), npoly, bits,
                                                         (uint32_t)bias & 0xFFFFu, reinterpret_cast<uint32_t*>(out),
                                                         in_range);
    return cudaGetLastError();
}

cudaError_t launch_agg_finish_pack(const RingCtx& c, const int32_t* partial, int64_t npoly, int bits, int bias, uint8_t* out,
                                   uint8_t* in_range, cudaStream_t st) {
    if (npoly <= 0) return cudaSuccess;
    if (bits < 1 || bits > 16) return cudaErrorInvalidValue;
    const uint32_t off = ((1u << 30) / c.m.q + 1) * c.m.q;
    k_agg_finish_pack<<<wire_grid(npoly, c.num_sms), WBS, 0, st>>>(c.m, off, partial, npoly, bits, (uint32_t)bias & 0xFFFFu,
                                                                    reinterpret_cast<uint32_t*>(out), in_range);
    return cudaGetLastError();
}

cudaError_t launch_addsub_packed(const RingCtx& c, const uint8_t* a, int a_bits, int a_bias, const uint8_t* b, int b_bits,
                                 int b_bias, int sub, int64_t npoly, int bits, int bias, uint8_t* out, uint8_t* in_range,
                                 cudaStream_t st) {
    if (npoly <= 0) return cudaSuccess;
    if (a_bits < 1 || a_bits > 16 || b_bits < 1 || b_bits > 16 || bits < 1 || bits > 16) return cudaErrorInvalidValue;
    k_addsub_packed<<<wire_grid(npoly, c.num_sms), WBS, 0, st>>>(
        c.m, reinterpret_cast<const uint32_t*>(a), a_bits, (uint32_t)a_bias & 0xFFFFu, reinterpret_cast<const uint32_t*>(b),
        b_bits, (uint32_t)b_bias & 0xFFFFu, sub, npoly, bits, (uint32_t)bias & 0xFFFFu, reinterpret_cast<uint32_t*>(out), in_range);
    return cudaGetLastError();
}

cudaError_t launch_unpack(const RingCtx& c, const uint8_t* in, int64_t npoly, int bits, int bias, void* out,
                          cudaStream_t st) {
    if (npoly <= 0) return cudaSuccess;
    if (bits < 1 || bits > 16) return cudaErrorInvalidValue;
    k_unpack<<<wire_grid(npoly, c.num_sms), WBS, 0, st>>>(reinterpret_cast<const uint32_t*>(in), npoly, bits,
                                                           (uint32_t)bias & 0xFFFFu, static_cast<uint16_t*>(out));
    return cudaGetLastError();
}

}  // namespace lcb
