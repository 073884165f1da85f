// content.cu — hash inputs of the content mode built on the device (sm_100a).
//
// In content mode (one_time_keys.set_content_str(True)) str() of a verification key / public statement is
//   '<' + name + ' ' + SHAKE256(name || le16(secpar) || centred int16 coefficient rows, little-endian).hexdigest(16) + '>'
// (57 bytes; name = OneTimeVerificationKey with rows left, right, or OneTimePublicStatement with one row).  Every
// challenge message and BKLM aggregation message contains such strings.  Three kernels make them from the engine's
// own arrays:
//   k_content_str         one SHAKE256 sponge per THREAD (lcb_device.cuh keccak_f1600); the coefficient rows of a
//                         block's 128 items are staged rate block by rate block through shared memory so that the
//                         warp's global loads read whole contiguous 136-byte spans instead of 128 rows 1 KB apart;
//   k_challenge_inputs    [st_str ', '] vk_str ', ' msg per item, one warp per item (byte copy, memory-bound);
//   k_aggregation_inputs  '[' + ', '.join("(" + vk_str + ", '" + msg + "')") + ']' per group, one warp per item at the
//                         offset the closed form of the group layout gives it.
#include "engine.h"

namespace lcb {

namespace {

constexpr int CBS = 128;                        // threads (sponges) per block of k_content_str
constexpr int CS_LANES = 17;                    // 64-bit lanes per 136-byte rate block
static __constant__ uint64_t c_rc[24] = LCB_KECCAK_RC_INIT;

__device__ __forceinline__ uint8_t hex_digit(uint32_t v) { return (uint8_t)(v < 10 ? '0' + v : 'a' + v - 10); }

// coef int16[n][rows][256] (centred, natural order) -> out uint8[n][57].  The sponge input of item i is the 24-byte
// prefix (name || le16(secpar), in `prefix` as three little-endian 64-bit lanes) followed by its 512*rows coefficient
// bytes; the prefix is a multiple of 8 bytes, so stream lane k >= 3 is lane k - 3 of the item's coefficient rows.
__global__ void __launch_bounds__(CBS) k_content_str(const uint2* __restrict__ coef, int64_t n, int rows, uint4 prefix_lo,
                                                     uint2 prefix_hi, uint4 head_lo, uint2 head_hi,
                                                     uint8_t* __restrict__ out) {
    __shared__ uint2 stage[CS_LANES][CBS + 1];   // [lane][sponge]: +1 keeps both the fill and the column reads conflict-free
    const int tid = threadIdx.x;
    const int64_t base = (int64_t)blockIdx.x * CBS;
    const int64_t cnt = n - base < CBS ? n - base : CBS;
    const int data_lanes = 64 * rows;
    const int tot_lane = 3 + data_lanes;                         // the 0x1F pad byte opens this lane (input bytes % 8 == 0)
    const int nblocks = (8 * tot_lane) / 136 + 1;
    const int last_lane = CS_LANES * nblocks - 1;                // the final 0x80 pad byte closes this lane
    const uint2 prefix[3] = {make_uint2(prefix_lo.x, prefix_lo.y), make_uint2(prefix_lo.z, prefix_lo.w), prefix_hi};
    KeccakState s;
#pragma unroll
    for (int i = 0; i < 25; ++i) { s.lo[i] = 0; s.hi[i] = 0; }
    for (int blk = 0; blk < nblocks; ++blk) {
        __syncthreads();                                         // the previous block's columns are consumed
        for (int k = tid; k < CS_LANES * CBS; k += CBS) {
            const int j = k / CS_LANES, w = k - j * CS_LANES;
            const int lane = CS_LANES * blk + w;
            uint2 v = make_uint2(0, 0);
            if (lane < 3) {
                v = prefix[lane];
            } else if (lane < tot_lane && j < cnt) {
                const int64_t at = (base + j) * data_lanes + (lane - 3);
                LCB_CHECK(base + j < n && lane - 3 < data_lanes);
                v = __ldg(coef + at);
            }
            if (lane == tot_lane) v.x ^= 0x1Fu;
            if (lane == last_lane) v.y ^= 0x80000000u;
            stage[w][j] = v;
        }
        __syncthreads();
#pragma unroll
        for (int i = 0; i < CS_LANES; ++i) {
            const uint2 v = stage[i][tid];
            s.lo[i] ^= v.x;
            s.hi[i] ^= v.y;
        }
        keccak_f1600(s, c_rc);
    }
    // 57 ASCII bytes per item, staged so that the block's output goes out as one contiguous run
    __syncthreads();
    uint8_t* ob = reinterpret_cast<uint8_t*>(&stage[0][0]);      // 128 * 57 = 7,296 bytes of the 17,544
    uint8_t* mine = ob + tid * 57;
    const uint32_t head[6] = {head_lo.x, head_lo.y, head_lo.z, head_lo.w, head_hi.x, head_hi.y};
#pragma unroll
    for (int b = 0; b < 24; ++b) mine[b] = (uint8_t)(head[b >> 2] >> (8 * (b & 3)));
    const uint32_t dg[4] = {s.lo[0], s.hi[0], s.lo[1], s.hi[1]};  // the first 16 squeezed bytes, little-endian lanes
#pragma unroll
    for (int b = 0; b < 16; ++b) {
        const uint32_t byte = (dg[b >> 2] >> (8 * (b & 3))) & 0xFFu;
        mine[24 + 2 * b] = hex_digit(byte >> 4);
        mine[25 + 2 * b] = hex_digit(byte & 15u);
    }
    mine[56] = '>';
    __syncthreads();
    uint8_t* o = out + base * 57;
    for (int k = tid; k < cnt * 57; k += CBS) {
        LCB_CHECK(base * 57 + k < n * 57);
        o[k] = ob[k];
    }
}

// item i -> out[out_off[i] ..): [st_str_i ', '] vk_str_i ', ' msg_i; out_off[i] = msg_off[i] - msg_off[0] + i * per.
// msg_i is msg[msg_off[i] - shift .. msg_off[i+1] - shift).
__global__ void __launch_bounds__(256) k_challenge_inputs(const uint8_t* __restrict__ st_str, const uint8_t* __restrict__ vk_str,
                                                          const uint8_t* __restrict__ msg, int64_t shift,
                                                          const int64_t* __restrict__ msg_off, int64_t n, int64_t out_len,
                                                          uint8_t* __restrict__ out, int64_t* __restrict__ out_off) {
    const int lane = threadIdx.x & 31;
    const int pre = st_str ? 59 : 0;
    const int per = pre + 59;
    const int64_t off0 = __ldg(msg_off);
    for (int64_t i = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; i < n; i += ((int64_t)gridDim.x * blockDim.x) >> 5) {
        const int64_t m0 = __ldg(msg_off + i), m1 = __ldg(msg_off + i + 1);
        const int64_t start = m0 - off0 + i * per, len = per + (m1 - m0);
        LCB_CHECK(m0 >= off0 && m1 >= m0 && start >= 0 && start + len <= out_len);
        if (lane == 0) {
            out_off[i] = start;
            if (i == n - 1) out_off[n] = start + len;
        }
        uint8_t* o = out + start;
        for (int64_t k = lane; k < len; k += 32) {
            uint8_t b;
            int64_t t = k;
            if (t < pre) {
                b = t < 57 ? st_str[i * 57 + t] : (t == 57 ? ',' : ' ');
            } else if ((t -= pre) < 59) {
                b = t < 57 ? vk_str[i * 57 + t] : (t == 57 ? ',' : ' ');
            } else {
                LCB_CHECK(m0 - shift + t - 59 >= 0);
                b = msg[m0 - shift + (t - 59)];
            }
            o[k] = b;
        }
    }
}

// Group g (sorted items agg_off[g] .. agg_off[g+1], gid[i] = group of item i) -> out[ag_off[g] .. ag_off[g+1]):
// '[' + ', '.join("(" + vk_str_i + ", '" + msg_i + "')") + ']'.  Item p of its group starts (after its ", " separator)
// at ag_off[g] + 1 + (msg_off[i] - msg_off[agg_off[g]]) + 65 p: 63 fixed bytes + the message + the separator per item.
__global__ void __launch_bounds__(256) k_aggregation_inputs(const int64_t* __restrict__ agg_off, const int64_t* __restrict__ ag_off,
                                                            int64_t n_agg, const int32_t* __restrict__ gid, int64_t total,
                                                            const uint8_t* __restrict__ vk_str, const uint8_t* __restrict__ msg,
                                                            int64_t shift, const int64_t* __restrict__ msg_off, int64_t out_len,
                                                            uint8_t* __restrict__ out) {
    const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x, nthreads = (int64_t)gridDim.x * blockDim.x;
    for (int64_t g = tid; g < n_agg; g += nthreads) {
        const int64_t a = __ldg(ag_off + g), b = __ldg(ag_off + g + 1);
        LCB_CHECK(a >= 0 && b >= a + 2 && b <= out_len);
        out[a] = '[';
        out[b - 1] = ']';
    }
    const int lane = threadIdx.x & 31;
    for (int64_t i = tid >> 5; i < total; i += nthreads >> 5) {
        const int g = __ldg(gid + i);
        LCB_CHECK(g >= 0 && g < n_agg);
        const int64_t first = __ldg(agg_off + g), p = i - first;
        const int64_t m0 = __ldg(msg_off + i), m1 = __ldg(msg_off + i + 1);
        const int64_t sep = p > 0 ? 2 : 0;
        const int64_t start = __ldg(ag_off + g) + 1 + (m0 - __ldg(msg_off + first)) + 65 * p - sep;
        const int64_t len = sep + 63 + (m1 - m0);
        LCB_CHECK(p >= 0 && m1 >= m0 && start >= 1 && start + len < out_len);
        uint8_t* o = out + start;
        for (int64_t k = lane; k < len; k += 32) {
            int64_t t = k - sep;
            uint8_t c;
            if (t < 0) c = t == -2 ? ',' : ' ';
            else if (t == 0) c = '(';
            else if (t < 58) c = vk_str[i * 57 + (t - 1)];
            else if (t < 61) c = t == 58 ? ',' : (t == 59 ? ' ' : '\'');
            else if ((t -= 61) < m1 - m0) c = msg[m0 - shift + t];
            else c = t == m1 - m0 ? '\'' : ')';
            o[k] = c;
        }
    }
}

int warp_grid(int64_t items, int num_sms) {
    const int64_t blocks = (items + 7) / 8;          // 8 warps per 256-thread block, one item per warp
    const int64_t cap = (int64_t)num_sms * 16;
    return (int)(blocks < 1 ? 1 : (blocks < cap ? blocks : cap));
}

}  // namespace

cudaError_t launch_content_str(const RingCtx& c, const int16_t* coef, int64_t n, int rows, const uint8_t (&prefix)[24],
                               const uint8_t (&head)[24], uint8_t* out, cudaStream_t st) {
    if (n <= 0) return cudaSuccess;
    if (rows < 1 || rows > 2) return cudaErrorInvalidValue;
    uint32_t p[6], h[6];
    for (int i = 0; i < 6; ++i) {
        p[i] = (uint32_t)prefix[4 * i] | (uint32_t)prefix[4 * i + 1] << 8 | (uint32_t)prefix[4 * i + 2] << 16 |
               (uint32_t)prefix[4 * i + 3] << 24;
        h[i] = (uint32_t)head[4 * i] | (uint32_t)head[4 * i + 1] << 8 | (uint32_t)head[4 * i + 2] << 16 |
               (uint32_t)head[4 * i + 3] << 24;
    }
    (void)c;
    k_content_str<<<(unsigned)((n + CBS - 1) / CBS), CBS, 0, st>>>(reinterpret_cast<const uint2*>(coef), n, rows,
                                                                 make_uint4(p[0], p[1], p[2], p[3]), make_uint2(p[4], p[5]),
                                                                 make_uint4(h[0], h[1], h[2], h[3]), make_uint2(h[4], h[5]), out);
    return cudaGetLastError();
}

cudaError_t launch_challenge_inputs(const RingCtx& c, const uint8_t* st_str, const uint8_t* vk_str, const uint8_t* msg,
                                    int64_t shift, const int64_t* msg_off, int64_t n, int64_t out_len, uint8_t* out,
                                    int64_t* out_off, cudaStream_t st) {
    if (n <= 0) return cudaSuccess;
    k_challenge_inputs<<<warp_grid(n, c.num_sms), 256, 0, st>>>(st_str, vk_str, msg, shift, msg_off, n, out_len, out, out_off);
    return cudaGetLastError();
}

cudaError_t launch_aggregation_inputs(const RingCtx& c, const int64_t* agg_off, const int64_t* ag_off, int64_t n_agg,
                                      const int32_t* gid, int64_t total, const uint8_t* vk_str, const uint8_t* msg,
                                      int64_t shift, const int64_t* msg_off, int64_t out_len, uint8_t* out, cudaStream_t st) {
    if (n_agg <= 0) return cudaSuccess;
    const int64_t work = total > n_agg / 32 ? total : n_agg / 32;
    k_aggregation_inputs<<<warp_grid(work, c.num_sms), 256, 0, st>>>(agg_off, ag_off, n_agg, gid, total, vk_str, msg, shift,
                                                                     msg_off, out_len, out);
    return cudaGetLastError();
}

}  // namespace lcb
