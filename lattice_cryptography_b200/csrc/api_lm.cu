// api_lm.cu — LM-OTS entry points of the C ABI: key generation (plain and packed), challenges, signing (plain, packed,
// from packed signing keys) and verification (plain, packed, packed adaptor pre-signatures).
#include <cstdlib>

#include "api_internal.h"

using namespace lcb;
using namespace lcb::abi;

namespace {

// host signatures are moved and verified 2^17 triples at a time (0.87 / 1.5 GB per chunk)
constexpr int64_t kPipeChunk = 1 << 17;

// The body of lcb_lm_keygen_batch (pk == null) and of lcb_lm_keygen_packed_batch (pk set, every unpacked output null).
int keygen(lcb_ctx* c, const lcb_scheme* sch, const uint8_t* seeds, const int64_t* seed_off, int64_t n, int16_t* sk_coef,
           uint16_t* sk_ntt, uint16_t* vk_ntt, int16_t* vk_coef, const PackedOut* pk, const char* name) {
    if (int st = need_key_ch(c, name)) return st;
    if (n == 0) return LCB_OK;
    CK(c, cudaSetDevice(c->device));
    const int l = c->l;
    SamplerArgs left{}, right{};
    int st = fill_sampler(c, left, salt_of(sch->sk_salt).c_str(), "LEFT", sch->sk_bd, sch->sk_wt, l);
    if (st == LCB_OK) st = fill_sampler(c, right, salt_of(sch->sk_salt).c_str(), "RIGHT", sch->sk_bd, sch->sk_wt, l);
    if (st != LCB_OK) return fail(c, st, "bad signing-key parameters");
    int64_t total = 0;
    CK(c, last_offset(c, seeds, seed_off, n, &total));
    Staging sg(c);
    const uint8_t* d_seeds = sg.in(seeds, (size_t)total);
    const int64_t* d_off = sg.in(seed_off, (size_t)n + 1);
    const size_t D_ = (size_t)c->d * ew(c);       // 16-bit units per polynomial (twice the degree in a wide context)
    int16_t* d_sk_coef = sg.out(sk_coef, (size_t)n * 2 * l * D_, true);
    uint16_t* d_sk_ntt = sg.out(sk_ntt, (size_t)n * 2 * l * D_, true);
    uint16_t* d_vk_ntt = sg.out(vk_ntt, (size_t)n * 2 * D_);
    int16_t* d_vk_coef = sg.out(vk_coef, (size_t)n * 2 * D_);
    uint8_t* d_skp = pk ? sg.out(pk->rows, (size_t)n * 2 * l * 32 * pk->bits, true) : nullptr;
    uint8_t* d_skr = pk ? sg.out(pk->in_range, (size_t)n * 2 * l) : nullptr;
    uint8_t* d_vkp = pk ? sg.out(pk->pub, (size_t)n * 2 * 32 * pk->pub_bits) : nullptr;
    CK(c, sg.status());
    if ((st = need_aligned4(c, {d_skp, d_vkp}))) return st;
    // Signing keys pass through HBM in coefficient form between the sampler and the row-vector
    // product; when the caller does not want them, a bounded scratch chunk is reused.
    // Both halves of a key come from ONE paired sampler launch (stream 2i = left, 2i+1 = right: twice the
    // parallelism for small batches, half the launches).  The chunk is eight full waves of sampler streams
    // (5 resident blocks of 128 streams per SM) = 378,880 keys = 5.0 GB (secpar 128) / 8.9 GB (secpar 256)
    // of scratch, so that every launch fills the machine and tails are rare (tools/keygen_chunk_sweep.py:
    // 2.12 M keys/s at secpar 128 against 2.02-2.08 M for two or four waves).
    left.paired = 1;
    std::memcpy(left.salt2, right.salt, sizeof(left.salt2));
    left.salt2_len = right.salt_len;
    const int64_t wave = (int64_t)c->ring.num_sms * 5 * 128;
    int64_t chunk = d_sk_coef ? n : (n < 4 * wave ? n : 4 * wave);
    if (const char* env = getenv("LCB_KEYGEN_CHUNK")) {            // tuning knob (keys per sampler launch)
        const int64_t v = atoll(env);
        if (v > 0 && !d_sk_coef) chunk = v < n ? v : n;
    }
    int16_t* scratch = d_sk_coef ? nullptr : sg.alloc<int16_t>((size_t)chunk * 2 * l * D_, true);
    // NTT-form verification keys of a chunk, to be packed
    uint16_t* vk_scratch = d_vkp ? sg.alloc<uint16_t>((size_t)chunk * 2 * D_) : nullptr;
    CK(c, sg.status());
    st = for_chunks(n, chunk, [&](int64_t start, int64_t cnt, int64_t) -> int {
        int16_t* skc = d_sk_coef ? d_sk_coef + start * 2 * l * D_ : scratch;
        if (sch->sk_wt < c->d) CK(c, cudaMemsetAsync(skc, 0, (size_t)cnt * 2 * l * D_ * sizeof(int16_t), c->stream));
        left.msgs = d_seeds;
        left.off = d_off + start;
        left.n = 2 * cnt;
        left.dense_stride = (int64_t)l * c->d;
        left.out_dense = skc;
        CK(c, sampler_scratch(c, left));
        CK(c, timed(c, K_SAMPLER, [&] { return launch_sampler(left, c->stream); }));
        uint16_t* o_sk = d_sk_ntt ? d_sk_ntt + start * 2 * l * D_ : nullptr;
        uint16_t* o_vk = d_vk_ntt ? d_vk_ntt + start * 2 * D_ : vk_scratch;
        int16_t* o_vkc = d_vk_coef ? d_vk_coef + start * 2 * D_ : nullptr;
        CK(c, timed(c, K_MATVEC, [&] {
            return c->generic ? g_launch_matvec(c->gen, skc, cnt * 2, o_sk, o_vk, o_vkc, c->stream)
                              : launch_matvec(c->ring, skc, cnt * 2, o_sk, o_vk, o_vkc, c->stream);
        }));
        if (d_skp)
            CK(c, timed(c, K_PACK, [&] {
                return launch_pack(c->ring, skc, cnt * 2 * l, pk->bits, pk->bias, d_skp + start * 2 * l * 32 * pk->bits,
                                   d_skr ? d_skr + start * 2 * l : nullptr, c->stream);
            }));
        if (d_vkp)
            CK(c, timed(c, K_PACK, [&] {
                return launch_pack(c->ring, vk_scratch, cnt * 2, pk->pub_bits, 0, d_vkp + start * 2 * 32 * pk->pub_bits, nullptr,
                                   c->stream);
            }));
        return LCB_OK;
    });
    if (st != LCB_OK) return st;
    CK(c, sg.finish());
    return LCB_OK;
}

// lcb_lm_verify_batch on packed verification keys and signatures, and on packed statements when st_packed is set
// (adaptor verify: the statement is added to the right-hand side, as st_ntt is).  The batch is processed in chunks of
// 2^18: challenge sampler -> k_verify reading the packed rows directly (the shipped 11/14- and 13/16-bit packings, with
// statements at the key width), or unpack -> challenge sampler -> k_verify for any other width (unpacked copies
// bounded to ~2 GB of scratch).  The caller has checked the arguments.
int verify_packed(lcb_ctx* c, const lcb_scheme* sch, const uint8_t* vk_packed, int vk_bits, const uint8_t* chmsg,
                  const int64_t* chmsg_off, const uint8_t* sig_packed, int sig_bits, int sig_bias, const uint8_t* st_packed,
                  int st_bits, int64_t n, int bd, int wt, uint8_t* verdict) {
    if (int st = need_wire(c)) return st;
    if (int st = need_key_ch(c, st_packed ? "lcb_adaptor_verify_packed_batch" : "lcb_lm_verify_packed_batch")) return st;
    if (int st = within_limit(c, n, "items in one verify call")) return st;
    if (n == 0) return LCB_OK;
    CK(c, cudaSetDevice(c->device));
    const int l = c->l;
    int64_t total = 0;
    CK(c, last_offset(c, chmsg, chmsg_off, n, &total));
    const int64_t chunk = n < 2 * kPipeChunk ? n : 2 * kPipeChunk;
    const size_t sig_row = (size_t)l * 32 * sig_bits;
    Staging sg(c);
    const uint8_t* d_vkp = sg.in(vk_packed, (size_t)n * 2 * 32 * vk_bits);
    const uint8_t* d_msg = sg.in(chmsg, (size_t)total);
    const int64_t* d_off = sg.in(chmsg_off, (size_t)n + 1);
    // packed signatures in HOST memory cross PCIe chunk by chunk under the kernels of the previous chunk
    std::vector<cudaEvent_t> arrived;
    const uint8_t* d_sigp = sg.in_piped(sig_packed, n, sig_row, chunk, arrived);
    const uint8_t* d_stp = st_packed ? sg.in(st_packed, (size_t)n * 32 * st_bits) : nullptr;
    uint8_t* d_verdict = sg.out(verdict, (size_t)n);
    CK(c, sg.status());
    if (int st = need_aligned4(c, {d_vkp, d_sigp, d_stp})) return st;
    // The two shipped packings (11/14 and 13/16 bits) are expanded inside k_verify; any other width is unpacked
    // into scratch first.
    // The fused route streams packed signature rows with 16-byte cp.async and reads 16-bit key slots with 128-bit
    // loads, so it needs 16-byte aligned buffers (staged host buffers always are); a caller-owned device buffer that
    // is only 4-byte aligned takes the unpack-first route instead of raising a sticky misaligned-address fault.
    // Statements are read like key halves: they must have the key width and, at 16 bits, 16-byte aligned rows.
    const bool fused = aligned16({d_sigp, vk_bits == 14 ? nullptr : d_vkp, vk_bits == 14 ? nullptr : d_stp}) &&
                       (!d_stp || st_bits == vk_bits) && ((sig_bits == 11 && vk_bits == 14) || (sig_bits == 13 && vk_bits == 16));
    uint16_t* d_vk = fused ? nullptr : sg.alloc<uint16_t>((size_t)chunk * 2 * D);
    int16_t* d_sig = fused ? nullptr : sg.alloc<int16_t>((size_t)chunk * l * D);
    uint16_t* d_st = fused || !d_stp ? nullptr : sg.alloc<uint16_t>((size_t)chunk * D);
    int16_t* d_pairs = sg.alloc<int16_t>((size_t)chunk * sch->ch_wt * 2);
    CK(c, sg.status());
    const int vbd = bd > 32767 ? 32767 : bd;
    int st = for_chunks(n, chunk, [&](int64_t first, int64_t m, int64_t k) -> int {
        if (fused) {
            int st = run_challenge(c, sch, d_msg, d_off + first, m, d_pairs);
            if (st != LCB_OK) return st;
            if (!arrived.empty()) CK(c, cudaStreamWaitEvent(c->stream, arrived[k], 0));
            CK(c, timed(c, K_VERIFY, [&] {
                return launch_verify_packed(c->ring, d_sigp + (size_t)first * sig_row, sig_bits, sig_bias,
                                            d_vkp + (size_t)first * 2 * 32 * vk_bits, vk_bits, d_pairs, sch->ch_wt, m, vbd, wt,
                                            d_verdict + first, c->stream, d_stp ? d_stp + (size_t)first * 32 * st_bits : nullptr);
            }));
            return LCB_OK;
        }
        CK(c, timed(c, K_UNPACK, [&] {
            return launch_unpack(c->ring, d_vkp + (size_t)first * 2 * 32 * vk_bits, m * 2, vk_bits, 0, d_vk, c->stream);
        }));
        if (d_stp)
            CK(c, timed(c, K_UNPACK, [&] {
                return launch_unpack(c->ring, d_stp + (size_t)first * 32 * st_bits, m, st_bits, 0, d_st, c->stream);
            }));
        if (!arrived.empty()) CK(c, cudaStreamWaitEvent(c->stream, arrived[k], 0));
        CK(c, timed(c, K_UNPACK, [&] {
            return launch_unpack(c->ring, d_sigp + (size_t)first * sig_row, m * l, sig_bits, sig_bias, d_sig, c->stream);
        }));
        int st = run_challenge(c, sch, d_msg, d_off + first, m, d_pairs);
        if (st != LCB_OK) return st;
        CK(c, timed(c, K_VERIFY, [&] {
            return launch_verify(c->ring, d_sig, d_vk, d_pairs, sch->ch_wt, nullptr, d_st, m, vbd, wt, d_verdict + first, c->stream);
        }));
        return LCB_OK;
    });
    if (st != LCB_OK) return st;
    CK(c, sg.finish());
    return LCB_OK;
}

// The body of lcb_lm_sign_packed_batch over device buffers (d_range nullable): lcb_lm_sign_batch -> lcb_pack_batch.  Fused
// route (11- or 13-bit rows, 16-byte aligned): k_sign writes the packed rows and in_range flags itself.  Anything else signs
// into int16 scratch and packs it with k_pack, in chunks.
int sign_packed(lcb_ctx* c, Staging& sg, const lcb_scheme* sch, const uint16_t* d_sk, const uint8_t* d_msg, const int64_t* d_off,
                int64_t n, int sig_bits, int sig_bias, uint8_t* d_sigp, uint8_t* d_range) {
    const int l = c->l;
    const size_t row = (size_t)32 * sig_bits;
    int16_t* d_pairs = sg.alloc<int16_t>((size_t)n * sch->ch_wt * 2);
    CK(c, sg.status());
    int st = run_challenge(c, sch, d_msg, d_off, n, d_pairs);
    if (st != LCB_OK) return st;
    // k_sign stores whole packed rows with 16-byte stores: a caller-owned device buffer that is only 4-byte aligned
    // takes the composed route
    if ((sig_bits == 11 || sig_bits == 13) && aligned16({d_sigp})) {
        CK(c, timed(c, K_SIGN, [&] {
            return launch_sign_packed(c->ring, d_sk, d_pairs, sch->ch_wt, n, sig_bits, sig_bias, d_sigp, d_range, c->stream);
        }));
        return LCB_OK;
    }
    const int64_t chunk = n < kWireChunkPoly / l ? n : kWireChunkPoly / l;
    int16_t* d_sig = sg.alloc<int16_t>((size_t)chunk * l * D);
    CK(c, sg.status());
    return for_chunks(n, chunk, [&](int64_t first, int64_t m, int64_t) -> int {
        CK(c, timed(c, K_SIGN, [&] {
            return launch_sign(c->ring, d_sk + (size_t)first * 2 * l * D, d_pairs + (size_t)first * sch->ch_wt * 2, sch->ch_wt, m,
                               d_sig, c->stream);
        }));
        CK(c, timed(c, K_PACK, [&] {
            return launch_pack(c->ring, d_sig, m * l, sig_bits, sig_bias, d_sigp + (size_t)first * l * row,
                               d_range ? d_range + (size_t)first * l : nullptr, c->stream);
        }));
        return LCB_OK;
    });
}

}  // namespace

extern "C" {

int lcb_lm_keygen_batch(lcb_ctx* c, const lcb_scheme* sch, const uint8_t* seeds, const int64_t* seed_off, int64_t n,
                        int16_t* sk_coef, uint16_t* sk_ntt, uint16_t* vk_ntt, int16_t* vk_coef) {
    LCB_RANGE();
    if (!c || !sch || !seed_off || n < 0) return LCB_ERR_INVALID;
    return keygen(c, sch, seeds, seed_off, n, sk_coef, sk_ntt, vk_ntt, vk_coef, nullptr, "lcb_lm_keygen_batch");
}

// lcb_lm_keygen_batch -> lcb_pack_batch (signing keys, coefficient form) and lcb_pack_batch (verification keys, bias 0), chunk
// by chunk inside the keygen loop: the 16-bit keys never leave engine scratch.
int lcb_lm_keygen_packed_batch(lcb_ctx* c, const lcb_scheme* sch, const uint8_t* seeds, const int64_t* seed_off, int64_t n,
                               int sk_bits, int sk_bias, uint8_t* sk_packed, uint8_t* sk_in_range, int vk_bits,
                               uint8_t* vk_packed) {
    LCB_RANGE();
    if (!c || !sch || !seed_off || n < 0 || (!sk_packed && !vk_packed) || !wire_args_ok(sk_bits, sk_bias) ||
        !wire_args_ok(vk_bits, 0))
        return LCB_ERR_INVALID;
    if (int st = need_wire(c)) return st;
    if (int st = within_limit(c, n, "items in one keygen call")) return st;
    const PackedOut pk{sk_bits, sk_bias, sk_packed, sk_packed ? sk_in_range : nullptr, vk_bits, vk_packed};
    return keygen(c, sch, seeds, seed_off, n, nullptr, nullptr, nullptr, nullptr, &pk, "lcb_lm_keygen_packed_batch");
}

int lcb_challenge_batch(lcb_ctx* c, const lcb_scheme* sch, const uint8_t* chmsg, const int64_t* chmsg_off, int64_t n,
                        int16_t* out_pairs) {
    LCB_RANGE();
    if (!c || !sch || !chmsg_off || !out_pairs || n < 0) return LCB_ERR_INVALID;
    if (n == 0) return LCB_OK;
    CK(c, cudaSetDevice(c->device));
    int64_t total = 0;
    CK(c, last_offset(c, chmsg, chmsg_off, n, &total));
    Staging sg(c);
    const uint8_t* d_msg = sg.in(chmsg, (size_t)total);
    const int64_t* d_off = sg.in(chmsg_off, (size_t)n + 1);
    int16_t* d_pairs = sg.out(out_pairs, (size_t)n * sch->ch_wt * 2 * ew(c));
    CK(c, sg.status());
    int st = run_challenge(c, sch, d_msg, d_off, n, d_pairs);
    if (st != LCB_OK) return st;
    CK(c, sg.finish());
    return LCB_OK;
}

int lcb_lm_sign_batch(lcb_ctx* c, const lcb_scheme* sch, const uint16_t* sk_ntt, const uint8_t* chmsg,
                      const int64_t* chmsg_off, int64_t n, int16_t* sig) {
    LCB_RANGE();
    if (!c || !sch || !sk_ntt || !chmsg_off || !sig || n < 0) return LCB_ERR_INVALID;
    if (n == 0) return LCB_OK;
    CK(c, cudaSetDevice(c->device));
    const int l = c->l;
    int64_t total = 0;
    CK(c, last_offset(c, chmsg, chmsg_off, n, &total));
    const size_t D_ = (size_t)c->d * ew(c);
    Staging sg(c);
    const uint16_t* d_sk = sg.in(sk_ntt, (size_t)n * 2 * l * D_, true);
    const uint8_t* d_msg = sg.in(chmsg, (size_t)total);
    const int64_t* d_off = sg.in(chmsg_off, (size_t)n + 1);
    int16_t* d_sig = sg.out(sig, (size_t)n * l * D_);
    int16_t* d_pairs = sg.alloc<int16_t>((size_t)n * sch->ch_wt * 2 * ew(c));
    CK(c, sg.status());
    int st = run_challenge(c, sch, d_msg, d_off, n, d_pairs);
    if (st != LCB_OK) return st;
    CK(c, timed(c, K_SIGN, [&] {
        return c->generic ? g_launch_sign(c->gen, d_sk, d_pairs, sch->ch_wt, n, d_sig, c->stream)
                          : launch_sign(c->ring, d_sk, d_pairs, sch->ch_wt, n, d_sig, c->stream);
    }));
    CK(c, sg.finish());
    return LCB_OK;
}

int lcb_lm_verify_batch(lcb_ctx* c, const lcb_scheme* sch, const uint16_t* vk_ntt, const uint8_t* chmsg,
                        const int64_t* chmsg_off, const int16_t* sig, const uint16_t* st_ntt, int64_t n, int bd,
                        int wt, uint8_t* verdict) {
    LCB_RANGE();
    if (!c || !sch || !vk_ntt || !chmsg_off || !sig || !verdict || n < 0 || bd < 0 || wt < 0) return LCB_ERR_INVALID;
    if (int st = need_key_ch(c, "lcb_lm_verify_batch")) return st;
    if (int st = within_limit(c, n, "items in one verify call")) return st;
    if (n == 0) return LCB_OK;
    CK(c, cudaSetDevice(c->device));
    const int l = c->l;
    int64_t total = 0;
    CK(c, last_offset(c, chmsg, chmsg_off, n, &total));
    const size_t D_ = (size_t)c->d * ew(c);
    Staging sg(c);
    const uint16_t* d_vk = sg.in(vk_ntt, (size_t)n * 2 * D_);
    const uint8_t* d_msg = sg.in(chmsg, (size_t)total);
    const int64_t* d_off = sg.in(chmsg_off, (size_t)n + 1);
    // Signatures in HOST memory (the bulk of the bytes) cross PCIe in chunks on the copy stream while the
    // sampler and verify kernels of the previous chunk run; everything else is one launch over the batch.
    std::vector<cudaEvent_t> arrived;
    const int16_t* d_sig = sg.in_piped(sig, n, (size_t)l * D_, kPipeChunk, arrived);
    const uint16_t* d_st = sg.in(st_ntt, (size_t)n * D_);
    uint8_t* d_verdict = sg.out(verdict, (size_t)n);
    int16_t* d_pairs = sg.alloc<int16_t>((size_t)n * sch->ch_wt * 2 * ew(c));
    CK(c, sg.status());
    const int vbd = bd > 32767 ? 32767 : bd;
    const int64_t chunk = arrived.empty() ? n : std::min(n, kPipeChunk);
    int st = for_chunks(n, chunk, [&](int64_t first, int64_t m, int64_t k) -> int {
        int16_t* pairs = d_pairs + (size_t)first * sch->ch_wt * 2 * ew(c);
        int st = run_challenge(c, sch, d_msg, d_off + first, m, pairs);
        if (st != LCB_OK) return st;
        if (!arrived.empty()) CK(c, cudaStreamWaitEvent(c->stream, arrived[k], 0));
        CK(c, timed(c, K_VERIFY, [&] {
            if (c->generic)
                return g_launch_verify(c->gen, d_sig + (size_t)first * l * D_, d_vk + (size_t)first * 2 * D_, pairs, sch->ch_wt,
                                       nullptr, d_st ? d_st + (size_t)first * D_ : nullptr, m, bd, wt, d_verdict + first, c->stream);
            return launch_verify(c->ring, d_sig + (size_t)first * l * D_, d_vk + (size_t)first * 2 * D_, pairs, sch->ch_wt,
                                 nullptr, d_st ? d_st + (size_t)first * D_ : nullptr, m, vbd, wt, d_verdict + first,
                                 c->stream);
        }));
        return LCB_OK;
    });
    if (st != LCB_OK) return st;
    CK(c, sg.finish());
    return LCB_OK;
}

int lcb_lm_verify_packed_batch(lcb_ctx* c, const lcb_scheme* sch, const uint8_t* vk_packed, int vk_bits,
                               const uint8_t* chmsg, const int64_t* chmsg_off, const uint8_t* sig_packed, int sig_bits,
                               int sig_bias, int64_t n, int bd, int wt, uint8_t* verdict) {
    LCB_RANGE();
    if (!c || !sch || !vk_packed || !chmsg_off || !sig_packed || !verdict || n < 0 || bd < 0 || wt < 0 ||
        !wire_args_ok(vk_bits, 0) || !wire_args_ok(sig_bits, sig_bias))
        return LCB_ERR_INVALID;
    return verify_packed(c, sch, vk_packed, vk_bits, chmsg, chmsg_off, sig_packed, sig_bits, sig_bias, nullptr, 0, n, bd,
                         wt, verdict);
}

int lcb_adaptor_verify_packed_batch(lcb_ctx* c, const lcb_scheme* sch, const uint8_t* vk_packed, int vk_bits,
                                    const uint8_t* chmsg, const int64_t* chmsg_off, const uint8_t* sig_packed,
                                    int sig_bits, int sig_bias, const uint8_t* st_packed, int st_bits, int64_t n, int bd,
                                    int wt, uint8_t* verdict) {
    LCB_RANGE();
    if (!c || !sch || !vk_packed || !chmsg_off || !sig_packed || !st_packed || !verdict || n < 0 || bd < 0 || wt < 0 ||
        !wire_args_ok(vk_bits, 0) || !wire_args_ok(sig_bits, sig_bias) || !wire_args_ok(st_bits, 0))
        return LCB_ERR_INVALID;
    return verify_packed(c, sch, vk_packed, vk_bits, chmsg, chmsg_off, sig_packed, sig_bits, sig_bias, st_packed, st_bits,
                         n, bd, wt, verdict);
}

int lcb_lm_sign_packed_batch(lcb_ctx* c, const lcb_scheme* sch, const uint16_t* sk_ntt, const uint8_t* chmsg,
                             const int64_t* chmsg_off, int64_t n, int sig_bits, int sig_bias, uint8_t* sig_packed,
                             uint8_t* in_range) {
    LCB_RANGE();
    if (!c || !sch || !sk_ntt || !chmsg_off || !sig_packed || n < 0 || !wire_args_ok(sig_bits, sig_bias))
        return LCB_ERR_INVALID;
    if (int st = need_wire(c)) return st;
    if (n == 0) return LCB_OK;
    CK(c, cudaSetDevice(c->device));
    const int l = c->l;
    int64_t total = 0;
    CK(c, last_offset(c, chmsg, chmsg_off, n, &total));
    Staging sg(c);
    const uint16_t* d_sk = sg.in(sk_ntt, (size_t)n * 2 * l * D, true);
    const uint8_t* d_msg = sg.in(chmsg, (size_t)total);
    const int64_t* d_off = sg.in(chmsg_off, (size_t)n + 1);
    uint8_t* d_sigp = sg.out(sig_packed, (size_t)n * l * 32 * sig_bits);
    uint8_t* d_range = sg.out(in_range, (size_t)n * l);
    CK(c, sg.status());
    if (int st = need_aligned4(c, {d_sigp})) return st;
    int st = sign_packed(c, sg, sch, d_sk, d_msg, d_off, n, sig_bits, sig_bias, d_sigp, d_range);
    if (st != LCB_OK) return st;
    CK(c, sg.finish());
    return LCB_OK;
}

// unpack -> lcb_ntt_fwd_batch -> lcb_lm_sign_packed_batch in one call.  Fused route (sign_sk_fused_applies: 7- / 8-bit keys,
// 11- / 13-bit signatures, monomial challenges; both packed buffers 16-byte aligned): k_sign_sk sums the rotations of the
// packed coefficient-form rows directly.  Anything else unpacks and transforms the keys into bounded secret scratch, chunk
// by chunk, and signs each chunk with the body of lcb_lm_sign_packed_batch.
int lcb_lm_sign_packed_sk_batch(lcb_ctx* c, const lcb_scheme* sch, const uint8_t* sk_packed, int sk_bits, int sk_bias,
                                const uint8_t* chmsg, const int64_t* chmsg_off, int64_t n, int sig_bits, int sig_bias,
                                uint8_t* sig_packed, uint8_t* in_range) {
    LCB_RANGE();
    if (!c || !sch || !sk_packed || !chmsg_off || !sig_packed || n < 0 || !wire_args_ok(sk_bits, sk_bias) ||
        !wire_args_ok(sig_bits, sig_bias))
        return LCB_ERR_INVALID;
    if (int st = need_wire(c)) return st;
    if (int st = within_limit(c, n, "items in one sign call")) return st;
    if (n == 0) return LCB_OK;
    CK(c, cudaSetDevice(c->device));
    const int l = c->l;
    int64_t total = 0;
    CK(c, last_offset(c, chmsg, chmsg_off, n, &total));
    const size_t sk_item = (size_t)2 * l * 32 * sk_bits, sig_item = (size_t)l * 32 * sig_bits;
    Staging sg(c);
    const uint8_t* d_skp = sg.in(sk_packed, (size_t)n * sk_item, true);
    const uint8_t* d_msg = sg.in(chmsg, (size_t)total);
    const int64_t* d_off = sg.in(chmsg_off, (size_t)n + 1);
    uint8_t* d_sigp = sg.out(sig_packed, (size_t)n * sig_item);
    uint8_t* d_range = sg.out(in_range, (size_t)n * l);
    CK(c, sg.status());
    if (int st = need_aligned4(c, {d_skp, d_sigp})) return st;
    int st;
    if (aligned16({d_skp, d_sigp}) && sign_sk_fused_applies(sk_bits, sig_bits, sch->ch_bd, sch->ch_wt)) {
        int16_t* d_pairs = sg.alloc<int16_t>((size_t)n * sch->ch_wt * 2);
        CK(c, sg.status());
        if ((st = run_challenge(c, sch, d_msg, d_off, n, d_pairs)) != LCB_OK) return st;
        CK(c, timed(c, K_SIGN, [&] {
            return launch_sign_sk_packed(c->ring, d_skp, sk_bits, sk_bias, d_pairs, sch->ch_bd, sch->ch_wt, n, sig_bits, sig_bias,
                                         d_sigp, d_range, c->stream);
        }));
    } else {
        const int64_t chunk = n < kWireChunkPoly / (2 * l) ? n : kWireChunkPoly / (2 * l);
        int16_t* d_coef = sg.alloc<int16_t>((size_t)chunk * 2 * l * D, true);
        uint16_t* d_ntt = sg.alloc<uint16_t>((size_t)chunk * 2 * l * D, true);
        CK(c, sg.status());
        st = for_chunks(n, chunk, [&](int64_t first, int64_t m, int64_t) -> int {
            CK(c, timed(c, K_UNPACK, [&] {
                return launch_unpack(c->ring, d_skp + (size_t)first * sk_item, m * 2 * l, sk_bits, sk_bias, d_coef, c->stream);
            }));
            CK(c, timed(c, K_NTT_FWD, [&] { return launch_ntt_fwd(c->ring, d_coef, m * 2 * l, d_ntt, c->stream); }));
            Staging chunk_sg(c);                 // the chunk's challenge pairs and int16 scratch go back to the pool after it
            return sign_packed(c, chunk_sg, sch, d_ntt, d_msg, d_off + first, m, sig_bits, sig_bias,
                               d_sigp + (size_t)first * sig_item, d_range ? d_range + (size_t)first * l : nullptr);
        });
        if (st != LCB_OK) return st;
    }
    CK(c, sg.finish());
    return LCB_OK;
}

}  // extern "C"
