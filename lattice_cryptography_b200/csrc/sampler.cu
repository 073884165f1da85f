// sampler.cu — SHAKE256 and the fused squeeze->decode samplers (sm_100a).
//
// Replaces lattice_algebra's binary_digest / decode2indices / decode2coef / decode2polycoefs /
// hash2polynomial / hash2polynomialvector (restated in oracle/lattice_algebra/__init__.py; call
// sites lm_one_time_sigs.py:70-91,142-160, adaptor_sigs.py:86-96, bklm_one_time_agg_sigs.py:81).
//
// One SHAKE256 stream per THREAD: the 1600-bit state lives in 50 registers and the permutation is
// pure LOP3/SHF work at the ALU-pipe issue limit.  The digest is never written to HBM: each
// 136-byte rate block is spilled to a per-thread column of shared memory ([word][thread],
// conflict-free because all threads of a warp consume the stream in lock-step) and read back by a
// big-endian bit cursor that feeds the index / coefficient decoder directly.
#include "engine.h"
#include "sampler_device.cuh"

namespace lcb {

namespace {

constexpr int SBS = 128;          // threads per block = SHAKE streams per block

// round constants split into even-bit / odd-bit halves (keccak_f1600_half)
struct Rc2Table {
    uint32_t v[2][24];      // [even-bit halves | odd-bit halves] of the round constants
};
constexpr uint32_t cx_even_bits(uint64_t x) {
    uint32_t r = 0;
    for (int i = 0; i < 32; ++i) r |= (uint32_t)((x >> (2 * i)) & 1u) << i;
    return r;
}
constexpr Rc2Table make_rc2() {
    constexpr uint64_t rc[24] = LCB_KECCAK_RC_INIT;
    Rc2Table t{};
    for (int i = 0; i < 24; ++i) { t.v[0][i] = cx_even_bits(rc[i]); t.v[1][i] = cx_even_bits(rc[i] >> 1); }
    return t;
}
static __constant__ Rc2Table c_keccak_rc2 = make_rc2();

// Absorb an input into a fresh state; leaves the state PERMUTED, i.e. its first 136 bytes are the
// first squeeze block.  `rate` is this block's [34][SBS] staging area in shared memory.
__device__ __forceinline__ void absorb(KeccakState& s, uint32_t* rate, int tid, const InputView& in) {
#pragma unroll
    for (int i = 0; i < 25; ++i) { s.lo[i] = 0; s.hi[i] = 0; }
    const int64_t tot = in.total();
    const int64_t nblocks = tot / 136 + 1;          // the pad byte always needs room
    const int64_t last = nblocks * 136 - 1;
    for (int64_t blk = 0; blk < nblocks; ++blk) {
        for (int w = 0; w < RATE_WORDS; ++w) rate[w * SBS + tid] = in.word_at(blk * RATE_WORDS + w, tot, last);
#pragma unroll
        for (int i = 0; i < 17; ++i) {
            s.lo[i] ^= rate[(2 * i) * SBS + tid];
            s.hi[i] ^= rate[(2 * i + 1) * SBS + tid];
        }
        keccak_f1600(s, c_keccak_rc);
    }
}

// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(SBS) k_shake256(const uint8_t* __restrict__ in, const int64_t* __restrict__ off,
                                                  int64_t n, uint8_t* __restrict__ out, int64_t out_len) {
    __shared__ uint32_t rate[RATE_WORDS * SBS];
    const int tid = threadIdx.x;
    const int64_t inst = (int64_t)blockIdx.x * SBS + tid;
    if (inst >= n) return;   // no block-level sync in this kernel
    InputView iv{nullptr, 0, in + off[inst], off[inst + 1] - off[inst]};
    KeccakState s;
    absorb(s, rate, tid, iv);
    const uint8_t* rb = reinterpret_cast<const uint8_t*>(rate);
    uint8_t* o = out + inst * out_len;
    int64_t produced = 0;
    while (produced < out_len) {
#pragma unroll
        for (int i = 0; i < 17; ++i) {
            rate[(2 * i) * SBS + tid] = s.lo[i];
            rate[(2 * i + 1) * SBS + tid] = s.hi[i];
        }
        for (int k = 0; k < 136 && produced < out_len; ++k, ++produced)
            o[produced] = rb[((k >> 2) * SBS + tid) * 4 + (k & 3)];
        if (produced < out_len) keccak_f1600(s, c_keccak_rc);
    }
}

// ------------------------------------------------------------------------------------------------
// Device-side expansion of host entropy into seed bitstrings (the unseeded keygen path, make_random_seed at
// lm_one_time_sigs.py:58-61, for batches): seed i = the first `secpar` bits, most significant bit of each byte first,
// of SHAKE256(secret[0..32) || le64(first + i)), written as the ASCII '0'/'1' string the reference hashes.
// One thread per seed; the 40-byte input and the <= 64-byte output each fit one rate block.
__global__ void __launch_bounds__(128) k_seed_expand(const uint8_t* __restrict__ secret, int64_t first, int64_t n, int secpar,
                                                     uint8_t* __restrict__ out) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    KeccakState s;
#pragma unroll
    for (int k = 0; k < 25; ++k) { s.lo[k] = 0; s.hi[k] = 0; }
    const uint32_t* sw = reinterpret_cast<const uint32_t*>(secret);       // engine-owned, 4-byte aligned copy
#pragma unroll
    for (int k = 0; k < 4; ++k) { s.lo[k] = __ldg(sw + 2 * k); s.hi[k] = __ldg(sw + 2 * k + 1); }
    const uint64_t ctr = (uint64_t)(first + i);
    s.lo[4] = (uint32_t)ctr;
    s.hi[4] = (uint32_t)(ctr >> 32);
    s.lo[5] ^= 0x1Fu;                  // SHAKE domain separation + first pad bit at byte 40
    s.hi[16] ^= 0x80000000u;           // last pad bit at byte 135
    keccak_f1600(s, c_keccak_rc);
    uint8_t* o = out + i * secpar;
    for (int b = 0; b < secpar; ++b) {
        const int byte = b >> 3, word = byte >> 3, sh = 8 * (byte & 7) + (7 - (b & 7));
        uint32_t w = 0;
#pragma unroll
        for (int k = 0; k < 8; ++k)
            if (k == word) w = sh < 32 ? s.lo[k] >> sh : s.hi[k] >> (sh - 32);
        o[b] = (uint8_t)('0' + (w & 1u));
    }
}

// ------------------------------------------------------------------------------------------------
// Fused SHAKE256 squeeze + decode2polycoefs (sampler_device.cuh), one stream per thread.
// Shared memory per block: ring [54][P] u32, bmap [8][P] u32, two modulus tables, the piece-weight table.
// P = streams (threads) per block; compile-time so that column addressing is shifts, not multiplies
#ifndef LCB_EXP_SAMPLER_STREAMS
#define LCB_EXP_SAMPLER_STREAMS 640          // streams resident per SM the sampler is compiled for
#endif
template <int P>
__global__ void __launch_bounds__(P, LCB_EXP_SAMPLER_STREAMS / P) k_sampler(SamplerArgs a) {   // 5 x 128 streams resident per SM
    extern __shared__ uint32_t smem[];
    uint32_t* ring = smem;                       // [RING_WORDS][P]
    uint32_t* bmap = ring + RING_WORDS * P;      // [8][P]   (directly after the ring, see StreamCols)
    uint32_t* mutab = bmap + 8 * P;
    uint32_t* r16tab = mutab + 260;
    uint8_t* wtab = reinterpret_cast<uint8_t*>(r16tab + 260);     // [257][pieces]
    const int pieces = weight_pieces(a.idx_bits, a.mag_bits);

    const int tid = threadIdx.x;
    const int64_t inst_raw = (int64_t)blockIdx.x * P + tid;
    const bool live = inst_raw < a.n;
    const int64_t inst = live ? inst_raw : a.n - 1;
    // the offsets of this stream's input are requested first, so that their latency hides behind the table fill
    const int64_t item = a.paired ? inst >> 1 : inst;
    const bool second = a.paired && (inst & 1);
    const int64_t msg_begin = __ldg(a.off + item), msg_end = __ldg(a.off + item + 1);
    load_mod_tables(a.mod_tab, mutab, r16tab, wtab, a.wt, a.bd, pieces);
    __syncthreads();

    const InputView iv{reinterpret_cast<const uint32_t*>(second ? a.salt2 : a.salt), second ? a.salt2_len : a.salt_len,
                       a.msgs + msg_begin, msg_end - msg_begin};
    const DecodeParams dp{a.bd, a.wt, a.vec_len, a.idx_bits, a.mag_bits, a.pad_bits};
    const StreamCols sc{ring + tid, bmap + tid, P, mutab, r16tab, wtab, pieces, a.idx_scratch + inst_raw, a.idx_stride};
    int16_t* dense = a.out_dense ? a.out_dense + inst * a.dense_stride : nullptr;
    uint32_t* pairs = a.out_pairs ? reinterpret_cast<uint32_t*>(a.out_pairs) + inst * a.vec_len * (int64_t)a.wt : nullptr;
    const int wt = a.wt;
    sample_stream(dp, iv, sc, [&](int poly, int e, int idx, int coef) {
        if (!live) return;
        if (dense) dense[(int64_t)poly * D + idx] = (int16_t)coef;
        if (pairs) pairs[(int64_t)poly * wt + e] = (uint32_t)idx | ((uint32_t)(uint16_t)(int16_t)coef << 16);
    });
}

// ------------------------------------------------------------------------------------------------
// The same sampler for any power-of-two degree 32 <= d <= 1024 (run-time geometry, 16-bit parked indices, Horner
// field reduction) and, with CT = int32_t, for coefficient bounds beyond int16 (moduli q >= 2^16).  Shared memory
// per block: ring [54][P], bmap [d/32][P], mutab [d + 1].
template <int P, typename CT>
__global__ void __launch_bounds__(P) k_sampler_g(SamplerArgs a) {
    extern __shared__ uint32_t smem[];
    const GeoAny geo{a.d, a.logd};
    uint32_t* ring = smem;                       // [RING_WORDS][P]
    uint32_t* bmap = ring + RING_WORDS * P;      // [d / 32][P]
    uint32_t* mutab = bmap + geo.words() * P;    // [d + 1]
    const int tid = threadIdx.x;
    const int64_t inst_raw = (int64_t)blockIdx.x * P + tid;
    const bool live = inst_raw < a.n;
    const int64_t inst = live ? inst_raw : a.n - 1;
    const int64_t item = a.paired ? inst >> 1 : inst;
    const bool second = a.paired && (inst & 1);
    const int64_t msg_begin = a.shared_msg ? 0 : __ldg(a.off + item), msg_end = a.shared_msg ? a.shared_len : __ldg(a.off + item + 1);
    fill_mod_tables(mutab, nullptr, a.wt, a.d);
    __syncthreads();
    // per-stream salts (BKLM aggregation coefficients with ag_wt > 1: ag_salt || decimal index, prepared by
    // k_index_salts) or the one or two warp-uniform salts of the call
    const uint32_t* salt_w = a.stream_salts ? reinterpret_cast<const uint32_t*>(a.stream_salts + inst * SALT_BYTES)
                                            : reinterpret_cast<const uint32_t*>(second ? a.salt2 : a.salt);
    const int salt_len = a.stream_salts ? (int)a.stream_salt_len[inst] : (second ? a.salt2_len : a.salt_len);
    const InputView iv{salt_w, salt_len, a.msgs + msg_begin, msg_end - msg_begin};
    const DecodeParams dp{a.bd, a.wt, a.vec_len, a.idx_bits, a.mag_bits, a.pad_bits};
    const StreamColsT<uint16_t> sc{ring + tid, bmap + tid, P, mutab, nullptr, nullptr, 0,
                                   reinterpret_cast<uint16_t*>(a.idx_scratch) + inst_raw, a.idx_stride};
    CT* dense = a.out_dense ? reinterpret_cast<CT*>(a.out_dense) + inst * a.dense_stride : nullptr;
    CT* pairs = a.out_pairs ? reinterpret_cast<CT*>(a.out_pairs) + inst * a.vec_len * (int64_t)a.wt * 2 : nullptr;
    const int wt = a.wt, d = a.d;
    SpongeFeed feed;
    sample_stream_t<GeoAny, uint16_t>(geo, dp, iv, sc, feed, [&](int poly, int e, int idx, int coef) {
        if (!live) return;
        if (dense) dense[(int64_t)poly * d + idx] = (CT)coef;
        if (pairs) {
            pairs[((int64_t)poly * wt + e) * 2] = (CT)idx;
            pairs[((int64_t)poly * wt + e) * 2 + 1] = (CT)coef;
        }
    });
}

// ------------------------------------------------------------------------------------------------
// Low-latency form for a HANDFUL of streams (a single key generation is two streams of 829 / 2,853 permutations:
// 7.8 / 20.8 ms when one thread squeezes and decodes everything, lm_one_time_sigs.py:64-97).  One block per stream:
//   warp 0        : the sponge on a lane pair (keccak_f1600_half: 110 instead of ~185 issue slots per round),
//                   digest written to a global scratch as little-endian stream words, progress published in shared memory;
//   warps 1 .. l  : ONE decoder lane each (its own warp, so that each has its own issue slots), polynomial p of the
//                   vector, whose bits start at digest byte p * nb - the l decoders run behind the producer instead of
//                   after it, so the stream costs about the sponge alone.
// d = 256, 16-bit outputs; chunk sizes nb that are not a multiple of 8 bytes fall back to k_sampler.
constexpr int COOP_MAX_POLYS = 23;       // the widest shipped vector (secpar 256); 24 warps per block

// decoder k runs in warp 1 + k + k / 3: warps 4, 8, 12, ... stay empty, because they would share warp 0's scheduler
// (warp id mod 4) and take issue slots from the sponge, which is the critical path
__host__ __device__ constexpr int coop_warps(int polys) { return 1 + polys + (polys + 2) / 3; }

__global__ void __launch_bounds__(32 * coop_warps(COOP_MAX_POLYS)) k_sampler_coop(SamplerArgs a, uint32_t* __restrict__ digest,
                                                                          int64_t digest_stride, int words_per_poly) {
    __shared__ uint32_t rc_sh[2][24];
    __shared__ volatile unsigned produced;
    extern __shared__ uint32_t smem[];                       // decoders: [RING_WORDS + 8][vec_len] columns, then tables
    const int nd = a.vec_len;                                // decoder warps
    uint32_t* ring = smem;
    uint32_t* bmap = ring + RING_WORDS * nd;
    uint32_t* mutab = bmap + 8 * nd;
    uint32_t* r16tab = mutab + 260;
    uint8_t* wtab = reinterpret_cast<uint8_t*>(r16tab + 260);
    const int pieces = weight_pieces(a.idx_bits, a.mag_bits);
    if (threadIdx.x < 48) rc_sh[threadIdx.x / 24][threadIdx.x % 24] = c_keccak_rc2.v[threadIdx.x / 24][threadIdx.x % 24];
    if (threadIdx.x == 0) produced = 0;
    load_mod_tables(a.mod_tab, mutab, r16tab, wtab, a.wt, a.bd, pieces);
    __syncthreads();
    const int64_t inst = blockIdx.x;                         // one block per stream
    const int64_t item = a.paired ? inst >> 1 : inst;
    const bool second = a.paired && (inst & 1);
    uint32_t* dg = digest + inst * digest_stride;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (warp == 0) {
        // ---- producer: absorb salt || message, then squeeze vec_len * words_per_poly (+ one window) words
        const unsigned odd = lane & 1u;
        const int64_t msg_begin = __ldg(a.off + item), msg_end = __ldg(a.off + item + 1);
        const InputView iv{reinterpret_cast<const uint32_t*>(second ? a.salt2 : a.salt), second ? a.salt2_len : a.salt_len,
                           a.msgs + msg_begin, msg_end - msg_begin};
        const int64_t tot = iv.total();
        const int64_t in_blocks = tot / 136 + 1, in_last = in_blocks * 136 - 1;
        const uint32_t* rc = rc_sh[odd];
        KeccakHalfRot rot;
        keccak_half_rot_init(rot, odd);
        KeccakHalf s;
#pragma unroll
        for (int i = 0; i < 25; ++i) s.a[i] = 0;
        for (int64_t blk = 0; blk < in_blocks; ++blk) {
#pragma unroll 1
            for (int i = 0; i < 17; ++i) {
                const int64_t g = blk * 17 + i;
                const uint64_t x = (uint64_t)iv.word_at(2 * g, tot, in_last) | ((uint64_t)iv.word_at(2 * g + 1, tot, in_last) << 32);
                const uint32_t hv = keccak_half_of(x, odd);
#pragma unroll
                for (int j = 0; j < 17; ++j)
                    if (j == i) s.a[j] ^= hv;
            }
            keccak_f1600_half<4>(s, rc, rot);
        }
        const unsigned total_words = (unsigned)(nd * words_per_poly) + RATE_WORDS + RING_EXTRA;
        unsigned blocks_out = 0;
        for (unsigned done = 0; done < total_words; done += RATE_WORDS) {
            // the lanes' state halves go out as they are ((even, odd) pair per sponge word); the decoders interleave
#pragma unroll
            for (int i = 0; i < 17; ++i)
                if (lane < 2) dg[done + 2 * i + odd] = s.a[i];
            // publish every fourth block (and the last): a device-wide fence costs hundreds of cycles of the critical path
            if ((++blocks_out & 3u) == 0 || done + RATE_WORDS >= total_words) {
                __threadfence();
                __syncwarp();
                if (lane == 0) produced = done + RATE_WORDS;
            }
            keccak_f1600_half<4>(s, rc, rot);
        }
    } else if ((warp & 3) != 0 && lane == 0 && warp - 1 - warp / 4 < nd) {
        // ---- decoder of polynomial p
        const int p = warp - 1 - warp / 4;
        const DecodeParams dp{a.bd, a.wt, 1, a.idx_bits, a.mag_bits, a.pad_bits};
        const StreamCols sc{ring + p, bmap + p, nd, mutab, r16tab, wtab, pieces,
                            a.idx_scratch + (inst * nd + p), a.idx_stride};
        BufferFeed feed{dg + (int64_t)p * words_per_poly, &produced, (unsigned)(p * words_per_poly), 0u};
        const InputView none{nullptr, 0, nullptr, 0};
        int16_t* dense = a.out_dense ? a.out_dense + inst * a.dense_stride + (int64_t)p * D : nullptr;
        uint32_t* pairs = a.out_pairs ? reinterpret_cast<uint32_t*>(a.out_pairs) + (inst * a.vec_len + p) * (int64_t)a.wt : nullptr;
        sample_stream_t<Geo256, uint8_t>(Geo256{}, dp, none, sc, feed, [&](int, int e, int idx, int coef) {
            if (dense) dense[idx] = (int16_t)coef;
            if (pairs) pairs[e] = (uint32_t)idx | ((uint32_t)(uint16_t)(int16_t)coef << 16);
        });
    }
}

// salt' = salt || decimal(first + i), zero padded to SALT_BYTES, one per stream (aggregation coefficients)
__global__ void k_index_salts(SamplerArgs a, uint8_t* __restrict__ salts, int32_t* __restrict__ lens) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= a.n) return;
    uint8_t* s = salts + i * SALT_BYTES;
    for (int b = 0; b < SALT_BYTES; ++b) s[b] = b < a.salt_len ? a.salt[b] : 0;
    uint64_t v = (uint64_t)(a.index_first + i);
    int nd = 1;
    for (uint64_t t = v; t >= 10; t /= 10) ++nd;
    for (int pos = a.salt_len + nd - 1; pos >= a.salt_len; --pos, v /= 10) s[pos] = (uint8_t)('0' + v % 10);
    lens[i] = a.salt_len + nd;
}

// ------------------------------------------------------------------------------------------------
// BKLM aggregation coefficients (bklm_one_time_agg_sigs.py:60-81), ag_wt = ag_bd = 1: coefficient i is
// +-X^k with k = first digest byte and sign = top bit of the second byte of
// SHAKE256(ag_salt || str(i) || agmsg).  Every stream absorbs the SAME O(N)-byte message behind a
// salt of 8..27 bytes, so the message cannot be pre-absorbed; each thread walks it with aligned
// 32-bit loads (warp-uniform addresses wherever the decimal index has the same number of digits)
// and funnel shifts.  N streams x ~N*124/136 permutations: the O(N^2) Keccak work of the reference.
constexpr int ABS = 64;   // threads per block (finer blocks balance the ~1 s streams over 148 SMs)

__global__ void __launch_bounds__(ABS) k_agg_coefs(SamplerArgs a) {
    __shared__ uint32_t edge[RATE_WORDS * ABS];
    const int64_t inst = (int64_t)blockIdx.x * ABS + threadIdx.x;
    if (inst >= a.n) return;
    // salt' = ag_salt || decimal(index), at most 27 bytes, kept in eight registers as words
    const uint64_t index = (uint64_t)(a.index_first + inst);
    uint32_t sw[8];
    const uint32_t* salt_w = reinterpret_cast<const uint32_t*>(a.salt);
#pragma unroll
    for (int i = 0; i < 8; ++i) sw[i] = i < (SALT_BYTES / 4) ? salt_w[i] : 0;
    int ndig = 1;
    for (uint64_t v = index; v >= 10; v /= 10) ++ndig;
    const int slen = a.salt_len + ndig;
    {
        uint64_t v = index;
        for (int dpos = slen - 1; dpos >= a.salt_len; --dpos, v /= 10) {
            const uint32_t ch = (uint32_t)('0' + (v % 10));
#pragma unroll
            for (int i = 0; i < 8; ++i)
                if ((dpos >> 2) == i) sw[i] |= ch << (8 * (dpos & 3));
        }
    }
    const int64_t tot = (int64_t)slen + a.shared_len;
    const int64_t nblocks = tot / 136 + 1;
    const int64_t last = nblocks * 136 - 1;
    const uint8_t* msg = a.msgs;
    auto salt_byte = [&](int p) -> uint32_t {
        uint32_t w = 0;
#pragma unroll
        for (int i = 0; i < 8; ++i)
            if ((p >> 2) == i) w = sw[i];
        return (w >> (8 * (p & 3))) & 0xFFu;
    };
    auto word_at = [&](int64_t k) -> uint32_t {
        const int64_t p = 4 * k;
        if (p >= slen && p + 4 <= tot) return load_u32_unaligned(msg + (p - slen));
        uint32_t v = 0;
#pragma unroll
        for (int b = 0; b < 4; ++b) {
            const int64_t q = p + b;
            uint32_t byte = q < slen ? salt_byte((int)q) : (q < tot ? (uint32_t)__ldg(msg + (q - slen)) : (q == tot ? 0x1Fu : 0u));
            if (q == last) byte ^= 0x80u;
            v |= byte << (8 * b);
        }
        return v;
    };
    KeccakState s;
#pragma unroll
    for (int i = 0; i < 25; ++i) { s.lo[i] = 0; s.hi[i] = 0; }
    for (int64_t blk = 0; blk < nblocks; ++blk) {
        const int64_t k0 = blk * RATE_WORDS;
        // interior blocks: every word is a plain unaligned message word
        const bool interior = 4 * k0 >= slen && 4 * (k0 + RATE_WORDS) <= tot;
        if (interior) {
            const uint8_t* p = msg + (4 * k0 - slen);
            const uintptr_t addr = reinterpret_cast<uintptr_t>(p);
            const uint32_t* w = reinterpret_cast<const uint32_t*>(addr & ~(uintptr_t)3);
            const unsigned sh = (unsigned)(addr & 3) * 8;
#ifdef LCB_CHECKED
            {   // the 34 or 35 aligned words of this block lie inside the (word-rounded) message
                const uintptr_t lo_ok = reinterpret_cast<uintptr_t>(msg) & ~(uintptr_t)3;
                const uintptr_t hi_ok = (reinterpret_cast<uintptr_t>(msg) + (uintptr_t)a.shared_len + 3) & ~(uintptr_t)3;
                LCB_CHECK(reinterpret_cast<uintptr_t>(w) >= lo_ok && reinterpret_cast<uintptr_t>(w + 34 + (sh ? 1 : 0)) <= hi_ok);
            }
#endif
            uint32_t prev = __ldg(w);
#pragma unroll
            for (int i = 0; i < 17; ++i) {
                const uint32_t m1 = __ldg(w + 2 * i + 1);
                const uint32_t m2 = (i < 16 || sh) ? __ldg(w + 2 * i + 2) : 0u;
                s.lo[i] ^= __funnelshift_r(prev, m1, sh);
                s.hi[i] ^= __funnelshift_r(m1, m2, sh);
                prev = m2;
            }
        } else {
            // first / last blocks (salt, tail, padding): assemble word by word through shared memory
            for (int w2 = 0; w2 < RATE_WORDS; ++w2) edge[w2 * ABS + threadIdx.x] = word_at(k0 + w2);
#pragma unroll
            for (int i = 0; i < 17; ++i) {
                s.lo[i] ^= edge[(2 * i) * ABS + threadIdx.x];
                s.hi[i] ^= edge[(2 * i + 1) * ABS + threadIdx.x];
            }
        }
        keccak_f1600(s, c_keccak_rc);
    }
    const uint32_t k = s.lo[0] & 0xFFu;                 // first digest byte: the 8 index bits
    const int sgn = (s.lo[0] >> 15) & 1u ? 1 : -1;      // top bit of the second byte: the sign bit
    reinterpret_cast<uint32_t*>(a.out_pairs)[inst] = k | ((uint32_t)(uint16_t)(int16_t)sgn << 16);
}

// One sponge of the derivation: SHAKE256(salt || decimal(index) || msg[0 .. msg_len)) -> packed (k, +-1) pair.
// The body of k_agg_coefs with the index, message and length as arguments (k_agg_coefs keeps its own copy: calling this
// from it reorders its prologue, and that kernel stays as measured).  `edge` is the block's [RATE_WORDS][ABS] staging.
__device__ __forceinline__ uint32_t agg_coef_pair(const SamplerArgs& a, uint64_t index, const uint8_t* msg, int64_t msg_len,
                                                  uint32_t* edge) {
    // salt' = ag_salt || decimal(index), at most 27 bytes, kept in eight registers as words
    uint32_t sw[8];
    const uint32_t* salt_w = reinterpret_cast<const uint32_t*>(a.salt);
#pragma unroll
    for (int i = 0; i < 8; ++i) sw[i] = i < (SALT_BYTES / 4) ? salt_w[i] : 0;
    int ndig = 1;
    for (uint64_t v = index; v >= 10; v /= 10) ++ndig;
    const int slen = a.salt_len + ndig;
    {
        uint64_t v = index;
        for (int dpos = slen - 1; dpos >= a.salt_len; --dpos, v /= 10) {
            const uint32_t ch = (uint32_t)('0' + (v % 10));
#pragma unroll
            for (int i = 0; i < 8; ++i)
                if ((dpos >> 2) == i) sw[i] |= ch << (8 * (dpos & 3));
        }
    }
    const int64_t tot = (int64_t)slen + msg_len;
    const int64_t nblocks = tot / 136 + 1;
    const int64_t last = nblocks * 136 - 1;
    auto salt_byte = [&](int p) -> uint32_t {
        uint32_t w = 0;
#pragma unroll
        for (int i = 0; i < 8; ++i)
            if ((p >> 2) == i) w = sw[i];
        return (w >> (8 * (p & 3))) & 0xFFu;
    };
    auto word_at = [&](int64_t k) -> uint32_t {
        const int64_t p = 4 * k;
        if (p >= slen && p + 4 <= tot) return load_u32_unaligned(msg + (p - slen));
        uint32_t v = 0;
#pragma unroll
        for (int b = 0; b < 4; ++b) {
            const int64_t q = p + b;
            uint32_t byte = q < slen ? salt_byte((int)q) : (q < tot ? (uint32_t)__ldg(msg + (q - slen)) : (q == tot ? 0x1Fu : 0u));
            if (q == last) byte ^= 0x80u;
            v |= byte << (8 * b);
        }
        return v;
    };
    KeccakState s;
#pragma unroll
    for (int i = 0; i < 25; ++i) { s.lo[i] = 0; s.hi[i] = 0; }
    for (int64_t blk = 0; blk < nblocks; ++blk) {
        const int64_t k0 = blk * RATE_WORDS;
        // interior blocks: every word is a plain unaligned message word
        const bool interior = 4 * k0 >= slen && 4 * (k0 + RATE_WORDS) <= tot;
        if (interior) {
            const uint8_t* p = msg + (4 * k0 - slen);
            const uintptr_t addr = reinterpret_cast<uintptr_t>(p);
            const uint32_t* w = reinterpret_cast<const uint32_t*>(addr & ~(uintptr_t)3);
            const unsigned sh = (unsigned)(addr & 3) * 8;
#ifdef LCB_CHECKED
            {   // the 34 or 35 aligned words of this block lie inside the (word-rounded) message
                const uintptr_t lo_ok = reinterpret_cast<uintptr_t>(msg) & ~(uintptr_t)3;
                const uintptr_t hi_ok = (reinterpret_cast<uintptr_t>(msg) + (uintptr_t)msg_len + 3) & ~(uintptr_t)3;
                LCB_CHECK(reinterpret_cast<uintptr_t>(w) >= lo_ok && reinterpret_cast<uintptr_t>(w + 34 + (sh ? 1 : 0)) <= hi_ok);
            }
#endif
            uint32_t prev = __ldg(w);
#pragma unroll
            for (int i = 0; i < 17; ++i) {
                const uint32_t m1 = __ldg(w + 2 * i + 1);
                const uint32_t m2 = (i < 16 || sh) ? __ldg(w + 2 * i + 2) : 0u;
                s.lo[i] ^= __funnelshift_r(prev, m1, sh);
                s.hi[i] ^= __funnelshift_r(m1, m2, sh);
                prev = m2;
            }
        } else {
            // first / last blocks (salt, tail, padding): assemble word by word through shared memory
            for (int w2 = 0; w2 < RATE_WORDS; ++w2) edge[w2 * ABS + threadIdx.x] = word_at(k0 + w2);
#pragma unroll
            for (int i = 0; i < 17; ++i) {
                s.lo[i] ^= edge[(2 * i) * ABS + threadIdx.x];
                s.hi[i] ^= edge[(2 * i + 1) * ABS + threadIdx.x];
            }
        }
        keccak_f1600(s, c_keccak_rc);
    }
    const uint32_t k = s.lo[0] & 0xFFu;                 // first digest byte: the 8 index bits
    const int sgn = (s.lo[0] >> 15) & 1u ? 1 : -1;      // top bit of the second byte: the sign bit
    return k | ((uint32_t)(uint16_t)(int16_t)sgn << 16);
}


// Many independent aggregates in one launch (lcb_bklm_aggregate_batch): stream i is local index j = i - agg_off[g] of
// group g = gid[i] and hashes ag_salt || str(j) || msg[msg_off[g] .. msg_off[g+1]).  One thread per sponge, as
// k_agg_coefs: the groups of the batch calls are short (the reference caps an aggregate at two signatures).
__global__ void __launch_bounds__(ABS) k_agg_coefs_seg(SamplerArgs a, const int32_t* __restrict__ gid,
                                                       const int64_t* __restrict__ agg_off, const int64_t* __restrict__ msg_off,
                                                       int64_t n_agg) {
    __shared__ uint32_t edge[RATE_WORDS * ABS];
    const int64_t inst = (int64_t)blockIdx.x * ABS + threadIdx.x;
    if (inst >= a.n) return;
    const int g = __ldg(gid + inst);
    LCB_CHECK(g >= 0 && g < n_agg);
    const int64_t j = inst - __ldg(agg_off + g);
    const int64_t m0 = __ldg(msg_off + g), m1 = __ldg(msg_off + g + 1);
    LCB_CHECK(j >= 0 && m0 <= m1);
    reinterpret_cast<uint32_t*>(a.out_pairs)[inst] = agg_coef_pair(a, (uint64_t)j, a.msgs + m0, m1 - m0, edge);
}

// gid[i] = group of sorted item i for i in [agg_off[g], agg_off[g+1]): one warp per group, lanes over its items
__global__ void __launch_bounds__(256) k_group_ids(const int64_t* __restrict__ agg_off, int64_t n_agg, int64_t total,
                                                   int32_t* __restrict__ gid) {
    const int lane = threadIdx.x & 31;
    for (int64_t g = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; g < n_agg; g += ((int64_t)gridDim.x * blockDim.x) >> 5) {
        const int64_t a0 = __ldg(agg_off + g), a1 = __ldg(agg_off + g + 1);
        LCB_CHECK(a0 >= 0 && a0 <= a1 && a1 <= total);
        for (int64_t i = a0 + lane; i < a1; i += 32) gid[i] = (int32_t)g;
    }
}

// ------------------------------------------------------------------------------------------------
// The same derivation with TWO lanes per sponge (keccak_f1600_half, lcb_device.cuh), for launches that would
// otherwise leave warp schedulers empty: on 8 GPUs a 2^16-signature aggregate is 8,192 streams per GPU = 256
// one-thread-per-sponge warps on 592 schedulers (0.39 of the Keccak roofline); as lane pairs it is 512 warps of
// half the length.  The message is common to all streams, so its 64-bit words are split into (even, odd) halves
// ONCE per salt-length phase by k_msg_interleave - a stream whose salt has slen bytes sees message byte
// 8 t + delta, delta = (-slen) mod 8, at the start of its word g0 + t - and an interior rate block is then 17
// aligned 32-bit loads and 17 XORs per lane (no funnel shifts at all; warp-uniform addresses wherever the
// decimal index has the same number of digits).

// il[delta][t] = (even, odd) halves of the little-endian 64-bit word msg[8 t + delta .. 8 t + delta + 8), for every t
// whose 8 bytes lie inside the message; grid.y = delta.
__global__ void __launch_bounds__(256) k_msg_interleave(const uint8_t* __restrict__ msg, int64_t len, uint2* __restrict__ il,
                                                        int64_t il_stride, unsigned delta_mask) {
    const int delta = blockIdx.y;
    if (!((delta_mask >> delta) & 1u)) return;
    const int64_t words = len >= delta ? (len - delta) / 8 : 0;
    for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < words; t += (int64_t)gridDim.x * blockDim.x) {
        const uint8_t* p = msg + 8 * t + delta;
        const uint64_t x = (uint64_t)load_u32_unaligned(p) | ((uint64_t)load_u32_unaligned(p + 4) << 32);
        il[delta * il_stride + t] = make_uint2(keccak_half_of(x, 0), keccak_half_of(x, 1));
    }
}

constexpr int ABS2 = 64;   // threads per block = 32 sponges

template <bool PREFETCH>
__global__ void __launch_bounds__(ABS2) k_agg_coefs_il(SamplerArgs a) {
    __shared__ uint32_t rc_sh[2][24];
    if (threadIdx.x < 48) rc_sh[threadIdx.x / 24][threadIdx.x % 24] = c_keccak_rc2.v[threadIdx.x / 24][threadIdx.x % 24];
    __syncthreads();
    const unsigned odd = threadIdx.x & 1u;
    const int64_t raw = ((int64_t)blockIdx.x * ABS2 + threadIdx.x) >> 1;
    const bool live = raw < a.n;
    const int64_t inst = live ? raw : a.n - 1;          // every lane stays in the shuffles
    const uint64_t index = (uint64_t)(a.index_first + inst);
    uint32_t sw[8];
    const uint32_t* salt_w = reinterpret_cast<const uint32_t*>(a.salt);
#pragma unroll
    for (int i = 0; i < 8; ++i) sw[i] = i < (SALT_BYTES / 4) ? salt_w[i] : 0;
    int ndig = 1;
    for (uint64_t v = index; v >= 10; v /= 10) ++ndig;
    const int slen = a.salt_len + ndig;
    {
        uint64_t v = index;
        for (int dpos = slen - 1; dpos >= a.salt_len; --dpos, v /= 10) {
            const uint32_t ch = (uint32_t)('0' + (v % 10));
#pragma unroll
            for (int i = 0; i < 8; ++i)
                if ((dpos >> 2) == i) sw[i] |= ch << (8 * (dpos & 3));
        }
    }
    const int64_t tot = (int64_t)slen + a.shared_len;
    const int64_t nblocks = tot / 136 + 1;
    const int64_t last = nblocks * 136 - 1;
    const uint8_t* msg = a.msgs;
    auto salt_byte = [&](int p) -> uint32_t {
        uint32_t w = 0;
#pragma unroll
        for (int i = 0; i < 8; ++i)
            if ((p >> 2) == i) w = sw[i];
        return (w >> (8 * (p & 3))) & 0xFFu;
    };
    auto word_at = [&](int64_t k) -> uint32_t {        // stream word k (bytes 4k .. 4k+3), SHAKE padding applied
        const int64_t p = 4 * k;
        if (p >= slen && p + 4 <= tot) return load_u32_unaligned(msg + (p - slen));
        uint32_t v = 0;
#pragma unroll
        for (int b = 0; b < 4; ++b) {
            const int64_t q = p + b;
            uint32_t byte = q < slen ? salt_byte((int)q) : (q < tot ? (uint32_t)__ldg(msg + (q - slen)) : (q == tot ? 0x1Fu : 0u));
            if (q == last) byte ^= 0x80u;
            v |= byte << (8 * b);
        }
        return v;
    };
    // stream word (64-bit) g is a plain message word iff g0 <= g < g0 + nl; it is then il[delta][g - g0]
    const int64_t g0 = (slen + 7) >> 3;
    const int delta = (int)(8 * g0 - slen);
    const int64_t nl = a.shared_len >= delta ? (a.shared_len - delta) / 8 : 0;
    const uint32_t* il = reinterpret_cast<const uint32_t*>(a.il_msg + delta * a.il_stride) + odd;
    const uint32_t* rc = rc_sh[odd];
    KeccakHalfRot rot;
    keccak_half_rot_init(rot, odd);
    KeccakHalf s;
#pragma unroll
    for (int i = 0; i < 25; ++i) s.a[i] = 0;
    // The lanes of a warp shuffle in lock-step, so the trip count is the warp's maximum (streams whose index has
    // one digit more may need one block more); a stream that is done keeps permuting, its result is taken on the way.
    const unsigned nb = (unsigned)(nblocks > 0xFFFFFFFFll ? 0xFFFFFFFFll : nblocks);
    const unsigned max_nb = __reduce_max_sync(0xFFFFFFFFu, nb);
    uint32_t result = 0;
    // The 17 message words of an interior block are requested one block AHEAD (before the permutation of the
    // previous block, volatile so that ptxas keeps them there): with one warp per scheduler nothing else would
    // cover the L2 round trip of a load issued at the top of the block.
    uint32_t pre[17];
    bool have = false;
    auto interior = [&](int64_t g) { return g >= g0 && g + 17 <= g0 + nl; };
    auto request = [&](int64_t g) {
        const uint32_t* w = il + 2 * (g - g0);
        LCB_CHECK(g - g0 >= 0 && g - g0 + 17 <= nl);
#pragma unroll
        for (int i = 0; i < 17; ++i) asm volatile("ld.global.nc.u32 %0, [%1];" : "=r"(pre[i]) : "l"(w + 2 * i));
    };
    for (unsigned blk = 0; blk < max_nb; ++blk) {
        const int64_t g = (int64_t)blk * 17;
        if (interior(g)) {
            if (!have) request(g);
#pragma unroll
            for (int i = 0; i < 17; ++i) s.a[i] ^= pre[i];
        } else {
            // first / last blocks (salt, tail, padding): assembled from bytes, split on the fly
#pragma unroll 1
            for (int i = 0; i < 17; ++i) {
                const uint64_t x = (uint64_t)word_at(2 * (g + i)) | ((uint64_t)word_at(2 * (g + i) + 1) << 32);
                const uint32_t h = keccak_half_of(x, odd);
#pragma unroll
                for (int j = 0; j < 17; ++j)
                    if (j == i) s.a[j] ^= h;
            }
        }
        have = PREFETCH && interior(g + 17);
        if (have) request(g + 17);
        keccak_f1600_half<12>(s, rc, rot);
        if (blk + 1 == nb) result = s.a[0];
    }
    // digest bits 0..7 (position) and 15 (sign) of word 0: even lane has bits 0,2,..,14, odd lane 1,3,..,15
    const uint32_t other = __shfl_xor_sync(0xFFFFFFFFu, result, 1);
    const uint32_t ev = odd ? other : result, od = odd ? result : other;
    uint32_t k = 0;
#pragma unroll
    for (int i = 0; i < 4; ++i) k |= ((ev >> i) & 1u) << (2 * i) | ((od >> i) & 1u) << (2 * i + 1);
    const int sgn = (od >> 7) & 1u ? 1 : -1;
    if (live && !odd) reinterpret_cast<uint32_t*>(a.out_pairs)[inst] = k | ((uint32_t)(uint16_t)(int16_t)sgn << 16);
}

}  // namespace

// The decoder tables for every modulus the fast decoder can meet (m <= 256): floor((2^32-1)/m), 2^16 mod m and the
// weights 2^(32k) mod m of the 32-bit pieces of a field (sampler_device.cuh: field_small).
void fill_sampler_mod_table(uint32_t* w) {
    for (int i = 0; i < SAMPLER_MOD_TABLE_WORDS; ++i) w[i] = 0;
    uint8_t* wt = reinterpret_cast<uint8_t*>(w + 520);
    for (uint32_t m = 1; m <= 256; ++m) {
        w[m] = 0xFFFFFFFFu / m;
        w[260 + m] = 65536u % m;
        if (m < 2) continue;
        const uint32_t r16 = 65536u % m, r32 = (r16 * r16) % m;
        uint32_t x = 1;
        for (int k = 0; k < WT_K; ++k) { wt[m * WT_K + k] = (uint8_t)x; x = (x * r32) % m; }
    }
}

cudaError_t launch_shake256(const uint8_t* in, const int64_t* off, int64_t n, uint8_t* out, int64_t out_len,
                            cudaStream_t st) {
    if (n <= 0) return cudaSuccess;
    int64_t blocks = (n + SBS - 1) / SBS;
    k_shake256<<<(unsigned)blocks, SBS, 0, st>>>(in, off, n, out, out_len);
    return cudaGetLastError();
}

cudaError_t launch_seed_expand(const uint8_t* secret, int64_t first, int64_t n, int secpar, uint8_t* out, cudaStream_t st) {
    if (n <= 0) return cudaSuccess;
    k_seed_expand<<<(unsigned)((n + 127) / 128), 128, 0, st>>>(secret, first, n, secpar, out);
    return cudaGetLastError();
}

cudaError_t launch_index_salts(const SamplerArgs& a, uint8_t* salts, int32_t* lens, cudaStream_t st) {
    if (a.n <= 0) return cudaSuccess;
    k_index_salts<<<(unsigned)((a.n + 127) / 128), 128, 0, st>>>(a, salts, lens);
    return cudaGetLastError();
}

static cudaError_t launch_sampler_generic(const SamplerArgs& a, cudaStream_t st) {
    constexpr int P = 64;
    if (!a.idx_scratch || a.idx_stride < (a.n + P - 1) / P * P) return cudaErrorInvalidValue;
    if (a.idx_bits > MAX_FIELD_BITS || 1 + a.mag_bits > MAX_FIELD_BITS) return cudaErrorInvalidValue;
    const size_t smem = (size_t)(RING_WORDS + a.d / 32) * P * 4 + (size_t)(a.d + 1) * 4;
    auto kern = a.wide ? k_sampler_g<P, int32_t> : k_sampler_g<P, int16_t>;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    kern<<<(unsigned)((a.n + P - 1) / P), P, smem, st>>>(a);
    return cudaGetLastError();
}

// Streams x polynomials-per-stream up to which the cooperative kernel (one block per stream) is used: below about one
// block per SM its latency advantage (the sponge alone instead of sponge + decoder on one thread) is what counts.
bool sampler_coop_applies(const SamplerArgs& a, int num_sms) {
    if (const char* env = getenv("LCB_SAMPLER_COOP")) { if (!atoi(env)) return false; }
    const int64_t bits = (int64_t)LOGD + (int64_t)(a.wt - 1) * a.idx_bits + (int64_t)a.wt * (1 + a.mag_bits) + a.pad_bits;
    return a.d == D && !a.wide && !a.stream_salts && !a.shared_msg && a.n <= num_sms && a.vec_len >= 2 &&
           a.vec_len <= COOP_MAX_POLYS && (bits / 8) % 8 == 0 && a.coop_digest != nullptr;     // chunks start on a 64-bit sponge word
}

static cudaError_t launch_sampler_coop(const SamplerArgs& a, cudaStream_t st) {
    const int64_t bits = (int64_t)LOGD + (int64_t)(a.wt - 1) * a.idx_bits + (int64_t)a.wt * (1 + a.mag_bits) + a.pad_bits;
    const int words_per_poly = (int)(bits / 32);
    const int pieces = weight_pieces(a.idx_bits, a.mag_bits);
    if (pieces > WT_K || a.idx_stride < a.n * a.vec_len) return cudaErrorInvalidValue;
    const size_t smem = (size_t)(RING_WORDS + 8) * a.vec_len * 4 + 2 * 260 * 4 + (size_t)(257 * pieces + 15) / 16 * 16;
    cudaError_t e = cudaFuncSetAttribute(k_sampler_coop, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    k_sampler_coop<<<(unsigned)a.n, 32 * coop_warps(a.vec_len), smem, st>>>(a, a.coop_digest, sampler_coop_digest_words(a.vec_len, words_per_poly),
                                                                     words_per_poly);
    return cudaGetLastError();
}

cudaError_t launch_sampler(const SamplerArgs& a, cudaStream_t st) {
    if (a.n <= 0) return cudaSuccess;
    if (a.d != D || a.wide || a.stream_salts || a.shared_msg) return launch_sampler_generic(a, st);
    if (a.coop_digest) return launch_sampler_coop(a, st);
    static int num_sms = 0;
    if (!num_sms) {
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&num_sms, cudaDevAttrMultiProcessorCount, dev);
    }
    // Grids under two full waves (5 resident 128-stream blocks per SM, register-limited) run as 64-stream blocks instead:
    // the ALU-bound streams then spread evenly (e.g. 2^16 streams: 6.92 blocks per SM, at most 7) instead
    // of leaving SMs with 3 blocks waiting for SMs with 4.
    const bool narrow = (a.n + SBS - 1) / SBS < (int64_t)num_sms * 10;
    const int threads = narrow ? SBS / 2 : SBS;
    if (!a.idx_scratch || a.idx_stride < (a.n + threads - 1) / threads * threads) return cudaErrorInvalidValue;
    const int pieces = weight_pieces(a.idx_bits, a.mag_bits);
    if (pieces > WT_K) return cudaErrorInvalidValue;
    size_t smem = (size_t)(RING_WORDS + 8) * threads * 4 + 2 * 260 * 4 + (size_t)(257 * pieces + 15) / 16 * 16;
    auto kern = narrow ? k_sampler<SBS / 2> : k_sampler<SBS>;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    int64_t blocks = (a.n + threads - 1) / threads;
    kern<<<(unsigned)blocks, threads, smem, st>>>(a);
    return cudaGetLastError();
}

// Which digit counts occur among the decimal indices [first, first + count)?  -> mask of the message phases
// delta = (-(salt_len + digits)) mod 8 the two-lane kernel will read.
unsigned agg_delta_mask(int salt_len, int64_t first, int64_t count) {
    auto digits = [](uint64_t v) { int n = 1; while (v >= 10) { v /= 10; ++n; } return n; };
    unsigned mask = 0;
    for (int d = digits((uint64_t)first); d <= digits((uint64_t)(first + count - 1)); ++d)
        mask |= 1u << ((8 - ((salt_len + d) & 7)) & 7);
    return mask;
}

bool agg_coefs_two_lane(int64_t n, int num_sms) {
    if (const char* env = getenv("LCB_AGG_LANES")) return atoi(env) == 2;       // tuning knob
    // Measured on B200 (tools/agg_coefs_timing.py; profiles/exp_r2_keccak_half_unroll.txt), one thread per sponge
    // against two lanes per sponge with 12 rounds per loop body and the next block requested a block ahead:
    // 8,192 streams 2.0 x, 16,384 streams 36.7 vs 36.3 ms, 24,576 streams 70.1 vs 53.6 ms, 32,768 streams 70.1 vs
    // 70.9 ms, 65,536 streams 3.55 vs 3.98 Gperm/s.  The finer grain never loses more than 1 %, so it is the default
    // at every size; the one-thread kernel stays for the comparison tests.
    (void)n;
    (void)num_sms;
    return true;
}

cudaError_t launch_agg_coefs(const SamplerArgs& a, int num_sms, cudaStream_t st) {
    if (a.n <= 0) return cudaSuccess;
    if (a.il_msg) {
        const unsigned mask = agg_delta_mask(a.salt_len, a.index_first, a.n);
        const int64_t words = a.shared_len / 8;
        if (words > 0) {
            int64_t need = (words + 255) / 256;
            dim3 grid((unsigned)(need < 4 * num_sms ? need : 4 * num_sms), 8);
            k_msg_interleave<<<grid, 256, 0, st>>>(a.msgs, a.shared_len, a.il_msg, a.il_stride, mask);
            cudaError_t e = cudaGetLastError();
            if (e != cudaSuccess) return e;
        }
        int64_t blocks = (2 * a.n + ABS2 - 1) / ABS2;
        // the next block is requested a block ahead (96 instead of 64 registers): with about one warp per scheduler
        // nothing else hides the load, and with many warps it still measured 1 - 2 % faster although only 2,960 of the
        // 4,096 warps of a 2^16-stream launch are then resident at once
        bool prefetch = true;
        if (const char* env = getenv("LCB_AGG_PREFETCH")) prefetch = atoi(env) != 0;
        auto kern = prefetch ? k_agg_coefs_il<true> : k_agg_coefs_il<false>;
        kern<<<(unsigned)blocks, ABS2, 0, st>>>(a);
        return cudaGetLastError();
    }
    int64_t blocks = (a.n + ABS - 1) / ABS;
    k_agg_coefs<<<(unsigned)blocks, ABS, 0, st>>>(a);
    return cudaGetLastError();
}

cudaError_t launch_group_ids(const int64_t* agg_off, int64_t n_agg, int64_t total, int32_t* gid, int num_sms, cudaStream_t st) {
    if (n_agg <= 0 || total <= 0) return cudaSuccess;
    const int64_t need = (n_agg + 7) / 8;                    // 8 warps (groups) per block
    k_group_ids<<<(unsigned)(need < 16 * num_sms ? need : 16 * num_sms), 256, 0, st>>>(agg_off, n_agg, total, gid);
    return cudaGetLastError();
}

cudaError_t launch_agg_coefs_seg(const SamplerArgs& a, const int32_t* gid, const int64_t* agg_off, const int64_t* msg_off,
                                 int64_t n_agg, cudaStream_t st) {
    if (a.n <= 0) return cudaSuccess;
    k_agg_coefs_seg<<<(unsigned)((a.n + ABS - 1) / ABS), ABS, 0, st>>>(a, gid, agg_off, msg_off, n_agg);
    return cudaGetLastError();
}

}  // namespace lcb
