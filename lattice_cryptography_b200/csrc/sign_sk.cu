// sign_sk.cu — LM sign / adaptor presign from PACKED COEFFICIENT-FORM signing keys straight into packed signatures
// (sm_100a; lcb_lm_sign_packed_sk_batch, the fused route).
//
// A packed signing key is uint8[2][l][32*sk_bits]: the rows of sk_left, then those of sk_right, in the wire format of
// wire.cu (v = (x + sk_bias) mod 2^16, sk_bits bits each).  The challenge c is ch_wt signed monomials (ch_bd = 1), so
// sig_i = sk_left_i ** c + sk_right_i is a signed sum of ch_wt negacyclic rotations of the row plus the right row - no
// transform at all (DESIGN.md §3.4).  One warp signs one item, row by row:
//
//   * Bytes, not coefficients.  With sk_bits <= 8 every packed field v fits a byte and x = v - sk_bias exactly (no
//     mod-2^16 wrap: v - sk_bias lies in [-32767, 255]).  The sum is taken over the raw fields and the bias is put back
//     once per position: sum_k s_k sigma_k(p) (v - bias), sigma = -1 on the wrapped reads.
//   * Parking.  The row is parked as E = [~v | v] (512 bytes, ~v = 255 - v): output p of the rotation by idx reads
//     E[256 + p - idx] whatever p and idx are (as k_agg_partial parks int16 rows).  A wrapped read returns 255 - v
//     instead of -v, so term k contributes s_k T - s_k (p >= idx_k ? bias : 255 - bias) with T the byte read.  Summed:
//       out[p] = sum_k s_k T_k(p) + corr[p] + x_right[p],   corr[p] = -bias S - (255 - 2 bias) W[p],
//       S = sum_k s_k,  W[p] = sum_{idx_k > p} s_k:
//     corr depends on the challenge only and is computed once per item (a histogram of the s_k and a warp suffix scan).
//   * Two values per add.  Lane j owns positions 4j..4j+3 and 128+4j..128+4j+3, i.e. one 32-bit word of bytes in each
//     half per term; the even and odd bytes of a word are split into two 16-bit lanes (one LOP / one PRMT) and added
//     into 32-bit accumulators that hold two positions each.  Positive and negative terms go to separate accumulators,
//     so every lane only ever adds bytes: a lane sum is at most ch_wt * 255 <= 256 * 255 < 2^16 - the accumulation is
//     exact for every ch_wt <= d, without a condition on the scheme beyond ch_bd = 1.
//   * Alignment copies.  The word a lane needs starts at byte 256 + 4j - idx, aligned only when idx = 0 mod 4.  The
//     parked row is written four times, copy r holding E[t + r] at byte t, so the term reads copy (-idx) mod 4 with
//     two conflict-free 32-bit loads (one shared-memory wavefront each) at immediate offsets 0 and 128 from one address.
//   * The exact result |out| <= (ch_wt + 1) * 32767 < 2^24 is reduced by Barrett reduction of out + off (off: a
//     multiple of q >= 2^30), centred, biased by sig_bias and packed exactly as sign_store_packed / k_pack write it.
#include "engine.h"

namespace lcb {

namespace {

constexpr int SKS_WARPS = 4;                   // warps (items in flight) per block
constexpr int SKS_TERMS = D + 8;               // challenge terms (ch_wt <= d), both sign lists padded to multiples of 4
constexpr int SKS_NULL = 4 * 512;              // byte offset (from the copies) of the zero row a padding term reads

struct SksWarp {
    uint32_t copies[4][128];                   // 4 alignment copies of the parked row E; reused to pack the output row
    uint32_t zero[64];                         // 256 zero bytes: the row of the padding terms
    int32_t hist[D];                           // sum of s_k per challenge index
    int32_t terms[SKS_TERMS];                  // byte offset of each term in `copies`: positives, pad, negatives, pad
};

// 16 packed SK_BITS-bit fields (starting at field 16 t of the row) as 16 bytes
template <int SK_BITS>
__device__ __forceinline__ void load_fields16(uint32_t (&e)[4], const uint32_t* __restrict__ row, int t) {
    if constexpr (SK_BITS == 8) {
        const uint4 v = __ldg(reinterpret_cast<const uint4*>(row) + t);
        e[0] = v.x; e[1] = v.y; e[2] = v.z; e[3] = v.w;
    } else {
        static_assert(SK_BITS == 7, "the fused route reads 7- and 8-bit keys");
        // fields 16t.. start at bit 112 t: word (7 t) / 2, shift 16 (t & 1); 112 + 16 bits fit the four words
        const uint32_t* p = row + ((7 * t) >> 1);
        const uint32_t sh = 16u * (t & 1);
        uint32_t w[5];
#pragma unroll
        for (int i = 0; i < 4; ++i) w[i] = __ldg(p + i);
        w[4] = 0;
        uint32_t a[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) a[i] = __funnelshift_r(w[i], w[i + 1], sh);
        // bytes m of the output word: fields 4m .. 4m + 3 = bits 28 m .. 28 m + 27 of the stream a
#pragma unroll
        for (int m = 0; m < 4; ++m) {
            const uint32_t g = __funnelshift_r(a[(28 * m) >> 5], a[((28 * m) >> 5) + 1], (28 * m) & 31);
            e[m] = (g & 0x7Fu) | ((g << 1) & 0x7F00u) | ((g << 2) & 0x7F0000u) | ((g << 3) & 0x7F000000u);
        }
    }
}

// fields 4 j .. 4 j + 3 (g = 0) or 128 + 4 j .. (g = 1) of a packed row as integers v
template <int SK_BITS>
__device__ __forceinline__ void load_fields4(int* v, const uint32_t* __restrict__ row, int j, int g) {
    const int bit = (128 * g + 4 * j) * SK_BITS;
    uint32_t w = __ldg(row + (bit >> 5));
    // 7 bits: the 28 bits of a group may straddle two words (never past the row's last word: the last group ends there)
    if constexpr (SK_BITS == 7) w = __funnelshift_r(w, (bit & 31) > 4 ? __ldg(row + (bit >> 5) + 1) : 0u, bit & 31);
#pragma unroll
    for (int b = 0; b < 4; ++b) v[b] = (int)((w >> (SK_BITS * b)) & ((1u << SK_BITS) - 1));
}

template <int SK_BITS, int SIG_BITS>
__global__ void __launch_bounds__(32 * SKS_WARPS) k_sign_sk(ModQ m, uint32_t off, int l, const uint8_t* __restrict__ sk_packed,
                                                            int sk_bias, const int16_t* __restrict__ ch_pairs, int ch_wt,
                                                            int64_t n, int sig_bias, uint8_t* __restrict__ sig_packed,
                                                            uint8_t* __restrict__ in_range) {
    __shared__ __align__(16) SksWarp ws[SKS_WARPS];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    SksWarp& w = ws[warp];
    const unsigned lt = (1u << lane) - 1u;
    for (int k = lane; k < 64; k += 32) w.zero[k] = 0;
    const unsigned char* cb = reinterpret_cast<const unsigned char*>(&w.copies[0][0]) + 4 * lane;   // + term offset
    constexpr int SK_ROW = 32 * SK_BITS, SK_WORDS = 8 * SK_BITS;
    const int bias = sk_bias;
    for (int64_t item = (int64_t)blockIdx.x * SKS_WARPS + warp; item < n; item += (int64_t)gridDim.x * SKS_WARPS) {
        // ---- the challenge: term offsets sorted by sign (each list padded with zero-row terms), corr[p]
        const uint32_t* pr = reinterpret_cast<const uint32_t*>(ch_pairs + item * ch_wt * 2);
        for (int k = lane; k < D; k += 32) w.hist[k] = 0;
        int npos = 0;
        for (int b = 0; b < ch_wt; b += 32)
            npos += __popc(__ballot_sync(0xFFFFFFFFu, b + lane < ch_wt && (int16_t)(__ldg(pr + b + lane) >> 16) > 0));
        const int p4 = (npos + 3) & ~3, nneg = ch_wt - npos, n4 = (nneg + 3) & ~3;
        __syncwarp();
        for (int b = 0, pos_before = 0, neg_before = 0; b < ch_wt; b += 32) {
            const bool valid = b + lane < ch_wt;
            const uint32_t pair = valid ? __ldg(pr + b + lane) : 0u;
            const int idx = (int)(pair & 0xFFu), s = (int)(int16_t)(pair >> 16);
            const unsigned bp = __ballot_sync(0xFFFFFFFFu, valid && s > 0), bn = __ballot_sync(0xFFFFFFFFu, valid && s <= 0);
            const int r = (-idx) & 3;
            const int term = r * 512 + (256 - idx - r);
            if (valid) {
                w.terms[s > 0 ? pos_before + __popc(bp & lt) : p4 + neg_before + __popc(bn & lt)] = term;
                atomicAdd(&w.hist[idx], s);
            }
            pos_before += __popc(bp);
            neg_before += __popc(bn);
        }
        if (lane < p4 - npos) w.terms[npos + lane] = SKS_NULL;
        if (lane < n4 - nneg) w.terms[p4 + nneg + lane] = SKS_NULL;
        __syncwarp();
        int corr[8];
        {
            const int4 ha = *reinterpret_cast<const int4*>(&w.hist[4 * lane]);
            const int4 hb = *reinterpret_cast<const int4*>(&w.hist[128 + 4 * lane]);
            const int ta = ha.x + ha.y + ha.z + ha.w, tb = hb.x + hb.y + hb.z + hb.w;
            int sa = ta, sb = tb;                                 // inclusive suffix sums over the lanes
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int ya = __shfl_down_sync(0xFFFFFFFFu, sa, o), yb = __shfl_down_sync(0xFFFFFFFFu, sb, o);
                if (lane + o < 32) { sa += ya; sb += yb; }
            }
            const int tot_b = __shfl_sync(0xFFFFFFFFu, sb, 0);
            const int S = __shfl_sync(0xFFFFFFFFu, sa, 0) + tot_b;
            const int above_a = sa - ta + tot_b, above_b = sb - tb;    // W at the last position of each group
            const int wv[8] = {ha.y + ha.z + ha.w + above_a, ha.z + ha.w + above_a, ha.w + above_a, above_a,
                               hb.y + hb.z + hb.w + above_b, hb.z + hb.w + above_b, hb.w + above_b, above_b};
#pragma unroll
            for (int i = 0; i < 8; ++i) corr[i] = -bias * S - (255 - 2 * bias) * wv[i];
        }
        // ---- the rows
        const uint32_t* key = reinterpret_cast<const uint32_t*>(sk_packed + item * 2 * l * SK_ROW);
        for (int i = 0; i < l; ++i) {
            const uint32_t* left = key + i * SK_WORDS;
            const uint32_t* right = key + (l + i) * SK_WORDS;
            uint32_t e[4];
            load_fields16<SK_BITS>(e, left, lane & 15);
            if (lane < 16) {
#pragma unroll
                for (int k = 0; k < 4; ++k) e[k] = ~e[k];
            }
            int xr[8];
            load_fields4<SK_BITS>(xr, right, lane, 0);
            load_fields4<SK_BITS>(xr + 4, right, lane, 1);
            const uint32_t nx = __shfl_down_sync(0xFFFFFFFFu, e[0], 1);   // lane 31: bytes past E, never read
#pragma unroll
            for (int r = 0; r < 4; ++r) {
                uint4 v;
                v.x = __funnelshift_r(e[0], e[1], 8 * r);
                v.y = __funnelshift_r(e[1], e[2], 8 * r);
                v.z = __funnelshift_r(e[2], e[3], 8 * r);
                v.w = __funnelshift_r(e[3], nx, 8 * r);
                reinterpret_cast<uint4*>(w.copies[r])[lane] = v;
            }
            __syncwarp();
            uint32_t pa_e = 0, pa_o = 0, pb_e = 0, pb_o = 0, na_e = 0, na_o = 0, nb_e = 0, nb_o = 0;
            const int4* tl = reinterpret_cast<const int4*>(w.terms);
            for (int k = 0; k < p4; k += 4) {
                const int4 t4 = tl[k >> 2];
                const int ts[4] = {t4.x, t4.y, t4.z, t4.w};
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    const uint32_t a = *reinterpret_cast<const uint32_t*>(cb + ts[u]);
                    const uint32_t b = *reinterpret_cast<const uint32_t*>(cb + ts[u] + 128);
                    pa_e += a & 0x00FF00FFu;
                    pa_o += __byte_perm(a, 0u, 0x4341);
                    pb_e += b & 0x00FF00FFu;
                    pb_o += __byte_perm(b, 0u, 0x4341);
                }
            }
            for (int k = p4; k < p4 + n4; k += 4) {
                const int4 t4 = tl[k >> 2];
                const int ts[4] = {t4.x, t4.y, t4.z, t4.w};
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    const uint32_t a = *reinterpret_cast<const uint32_t*>(cb + ts[u]);
                    const uint32_t b = *reinterpret_cast<const uint32_t*>(cb + ts[u] + 128);
                    na_e += a & 0x00FF00FFu;
                    na_o += __byte_perm(a, 0u, 0x4341);
                    nb_e += b & 0x00FF00FFu;
                    nb_o += __byte_perm(b, 0u, 0x4341);
                }
            }
            __syncwarp();                                         // the copies now stage the output row
            // positions 4j + {0, 1, 2, 3}: even bytes in the low / high halves of *_e, odd bytes in those of *_o
            const int sum[8] = {(int)(pa_e & 0xFFFFu) - (int)(na_e & 0xFFFFu), (int)(pa_o & 0xFFFFu) - (int)(na_o & 0xFFFFu),
                                (int)(pa_e >> 16) - (int)(na_e >> 16), (int)(pa_o >> 16) - (int)(na_o >> 16),
                                (int)(pb_e & 0xFFFFu) - (int)(nb_e & 0xFFFFu), (int)(pb_o & 0xFFFFu) - (int)(nb_o & 0xFFFFu),
                                (int)(pb_e >> 16) - (int)(nb_e >> 16), (int)(pb_o >> 16) - (int)(nb_o >> 16)};
            uint32_t v16[8];
#pragma unroll
            for (int b = 0; b < 8; ++b) {
                const int x = sum[b] + corr[b] + (xr[b] - bias);
                v16[b] = ((uint32_t)center(barrett_full((uint32_t)x + off, m), m) + (uint32_t)sig_bias) & 0xFFFFu;
            }
            uint32_t* stage = w.copies[0];                        // 256 biased values, natural order
            *reinterpret_cast<uint2*>(stage + 2 * lane) = make_uint2(v16[0] | (v16[1] << 16), v16[2] | (v16[3] << 16));
            *reinterpret_cast<uint2*>(stage + 64 + 2 * lane) = make_uint2(v16[4] | (v16[5] << 16), v16[6] | (v16[7] << 16));
            __syncwarp();
            // lane j packs values 8 j .. 8 j + 7 into SIG_BITS whole bytes at byte j * SIG_BITS of the packed row
            const uint4 q8 = *reinterpret_cast<const uint4*>(stage + 4 * lane);
            const uint32_t qw[4] = {q8.x, q8.y, q8.z, q8.w};
            uint8_t* rowb = reinterpret_cast<uint8_t*>(w.copies[1]);
            constexpr uint32_t LIMIT = 1u << SIG_BITS;
            bool ok = true;
            uint64_t acc = 0;
            int fill = 0, nb = 0;
#pragma unroll
            for (int b = 0; b < 8; ++b) {
                const uint32_t v = (qw[b >> 1] >> (16 * (b & 1))) & 0xFFFFu;
                ok = ok && v < LIMIT;
                acc |= (uint64_t)(v & (LIMIT - 1)) << fill;
                fill += SIG_BITS;
                while (fill >= 8) {
                    rowb[lane * SIG_BITS + nb++] = (uint8_t)acc;
                    acc >>= 8;
                    fill -= 8;
                }
            }
            ok = __all_sync(0xFFFFFFFFu, ok);
            __syncwarp();
            const int64_t row = item * l + i;
            LCB_CHECK(row < n * l);
            uint4* dst = reinterpret_cast<uint4*>(sig_packed + row * (32 * SIG_BITS));
            if (lane < 2 * SIG_BITS) dst[lane] = reinterpret_cast<const uint4*>(rowb)[lane];
            if (in_range && lane == 0) in_range[row] = ok ? 1 : 0;
            __syncwarp();                                         // the copies belong to the next row again
        }
    }
}

template <int SK_BITS, int SIG_BITS>
cudaError_t launch_sign_sk_t(const RingCtx& c, const uint8_t* sk_packed, int sk_bias, const int16_t* ch_pairs, int ch_wt,
                             int64_t n, int sig_bias, uint8_t* sig_packed, uint8_t* in_range, cudaStream_t st) {
    int nb = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, k_sign_sk<SK_BITS, SIG_BITS>, 32 * SKS_WARPS, 0) != cudaSuccess ||
        nb < 1)
        nb = 1;
    const int64_t need = (n + SKS_WARPS - 1) / SKS_WARPS, cap = (int64_t)c.num_sms * nb;
    const unsigned grid = (unsigned)(need < cap ? need : cap);
    const uint32_t off = ((1u << 30) / c.m.q + 1) * c.m.q;
    k_sign_sk<SK_BITS, SIG_BITS><<<grid, 32 * SKS_WARPS, 0, st>>>(c.m, off, c.l, sk_packed, sk_bias, ch_pairs, ch_wt, n,
                                                                 sig_bias, sig_packed, in_range);
    return cudaGetLastError();
}

}  // namespace

cudaError_t launch_sign_sk_packed(const RingCtx& c, const uint8_t* sk_packed, int sk_bits, int sk_bias,
                                  const int16_t* ch_pairs, int ch_bd, int ch_wt, int64_t n, int sig_bits, int sig_bias,
                                  uint8_t* sig_packed, uint8_t* in_range, cudaStream_t st) {
    if (n <= 0) return cudaSuccess;
    if (!sign_sk_fused_applies(sk_bits, sig_bits, ch_bd, ch_wt)) return cudaErrorNotSupported;
    if (sk_bits == 7 && sig_bits == 11)
        return launch_sign_sk_t<7, 11>(c, sk_packed, sk_bias, ch_pairs, ch_wt, n, sig_bias, sig_packed, in_range, st);
    if (sk_bits == 7)
        return launch_sign_sk_t<7, 13>(c, sk_packed, sk_bias, ch_pairs, ch_wt, n, sig_bias, sig_packed, in_range, st);
    if (sig_bits == 11)
        return launch_sign_sk_t<8, 11>(c, sk_packed, sk_bias, ch_pairs, ch_wt, n, sig_bias, sig_packed, in_range, st);
    return launch_sign_sk_t<8, 13>(c, sk_packed, sk_bias, ch_pairs, ch_wt, n, sig_bias, sig_packed, in_range, st);
}

}  // namespace lcb
