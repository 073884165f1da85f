// engine.h — host-side declarations shared by the C ABI files (api*.cu) and the kernel files (sampler.cu, ring.cu, ...).
#pragma once
#include <cstdint>
#include <cuda_runtime.h>
#include "lcb_device.cuh"

namespace lcb {

constexpr int SALT_BYTES = 48;

struct SamplerArgs {
    const uint8_t* msgs;       // ragged items (device)
    const int64_t* off;        // [n+1] (device); ignored when shared_msg
    int64_t n;
    int64_t shared_len;        // shared_msg: every instance hashes msgs[0 .. shared_len)
    int64_t index_first;       // shared_msg: decimal index appended to the salt = index_first + i
    int shared_msg;
    alignas(8) uint8_t salt[SALT_BYTES];
    int salt_len;
    // paired mode (key generation): stream j hashes item j >> 1 under salt (j even) or salt2 (j odd), so the two
    // halves of a key are sampled by ONE launch of 2 * items streams; n counts streams
    alignas(8) uint8_t salt2[SALT_BYTES];
    int salt2_len;
    int paired;
    int secpar, bd, wt, vec_len;
    int idx_bits;              // LOGD + secpar
    int mag_bits;              // btd - 1
    int pad_bits;              // 8*nb - bti - wt*btd
    int16_t* out_dense;        // or nullptr; instance stride below (elements)
    int64_t dense_stride;
    int16_t* out_pairs;        // or nullptr; [n][vec_len][wt][2]
    uint8_t* idx_scratch;      // device scratch, sampler_scratch_bytes(n, wt) bytes
    int64_t idx_stride;        // streams rounded up to whole blocks
    // shared_msg, two lanes per sponge: the message split into (even, odd) bit halves per 64-bit word, one copy per
    // byte phase delta = 0..7 (il_msg[delta * il_stride + t] <-> message bytes 8t + delta ..); nullptr = one thread
    // per sponge
    uint2* il_msg;
    int64_t il_stride;
    // ring geometry (d = 256 and 16-bit outputs take the fast kernel, anything else k_sampler_g)
    int d, logd;
    int wide;                  // outputs are int32 (moduli q >= 2^16) instead of int16
    // per-stream salts (aggregation coefficients with ag_wt > 1): [n][SALT_BYTES] bytes + [n] lengths, or nullptr
    const uint8_t* stream_salts;
    const int32_t* stream_salt_len;
    // cooperative low-latency kernel (few streams): digest scratch, sampler_coop_digest_words() words per stream;
    // nullptr = the ordinary one-thread-per-stream kernel
    uint32_t* coop_digest;
    // the decoder's modulus tables for every m <= 256 (sampler_mod_table_words() words, made once per context by
    // fill_sampler_mod_table): floor((2^32-1)/m) [260] | 2^16 mod m [260] | bytes 2^(32k) mod m [257][20]
    const uint32_t* mod_tab;
};
constexpr int SAMPLER_MOD_TABLE_WORDS = 260 + 260 + (257 * 20 + 3) / 4;
void fill_sampler_mod_table(uint32_t* host_words);      // SAMPLER_MOD_TABLE_WORDS words

cudaError_t launch_sampler(const SamplerArgs& a, cudaStream_t st);
cudaError_t launch_seed_expand(const uint8_t* secret, int64_t first, int64_t n, int secpar, uint8_t* out, cudaStream_t st);
bool sampler_coop_applies(const SamplerArgs& a, int num_sms);     // with a.coop_digest set to any non-null value
inline int64_t sampler_coop_digest_words(int vec_len, int words_per_poly) {
    return ((int64_t)vec_len * words_per_poly + 34 + 20 + 34 + 63) / 64 * 64;      // + one window and one block of slack
}
cudaError_t launch_index_salts(const SamplerArgs& a, uint8_t* salts, int32_t* lens, cudaStream_t st);
inline int64_t sampler_stride(int64_t n) { return (n + 127) / 128 * 128; }
// parked indices: one byte each for d = 256, two bytes on the generic path
inline size_t sampler_scratch_bytes(int64_t n, int wt, bool generic = false) {
    return (size_t)sampler_stride(n) * (size_t)wt * (generic ? 2 : 1);
}
cudaError_t launch_shake256(const uint8_t* in, const int64_t* off, int64_t n, uint8_t* out, int64_t out_len,
                            cudaStream_t st);
// shared-message fast path, wt == 1; two lanes per sponge when a.il_msg is set (see agg_coefs_two_lane)
cudaError_t launch_agg_coefs(const SamplerArgs& a, int num_sms, cudaStream_t st);
bool agg_coefs_two_lane(int64_t n, int num_sms);
inline int64_t agg_il_stride(int64_t msg_len) { return msg_len / 8 + 1; }
inline size_t agg_il_bytes(int64_t msg_len) { return (size_t)8 * (size_t)agg_il_stride(msg_len) * sizeof(uint2); }
// batches of independent aggregates (lcb_bklm_aggregate_batch): gid[i] = group of sorted item i, built once per call
// and shared by the segmented kernels; the coefficient of item i is H2P(salt || str(i - agg_off[g]) || message g)
cudaError_t launch_group_ids(const int64_t* agg_off, int64_t n_agg, int64_t total, int32_t* gid, int num_sms, cudaStream_t st);
cudaError_t launch_agg_coefs_seg(const SamplerArgs& a, const int32_t* gid, const int64_t* agg_off, const int64_t* msg_off,
                                 int64_t n_agg, cudaStream_t st);

// ---- generic degree / modulus (ring_generic.cu) -------------------------------------------------------------
struct GenRing {
    uint32_t q, half;          // modulus (< 2^31), (q - 1) / 2
    int d, logd;               // power-of-two degree 32..1024
    uint64_t mu64;             // floor(2^64 / q): 64-bit Barrett constant
    uint64_t pos_off;          // least multiple of q >= 2^31: makes any int32 coefficient non-negative
    uint32_t dinv, dinv_s;     // d^-1 mod q and its Shoup companion
    const uint32_t *w, *ws, *iw, *iws;   // device, [d]: zetas[k] = psi^bitrev_logd(k), inverses, Shoup companions
    const uint32_t* pw;        // device, [2d]: psi^e
};

struct GenCtx {
    GenRing r;
    const uint32_t* a_hat;     // device, uint32[l][d]: NTT(key_ch)
    int l, num_sms;
    bool wide;                 // int32 / uint32 element formats (q >= 2^16)
};

cudaError_t g_launch_ntt_fwd(const GenCtx& c, const void* coef, int64_t npoly, void* out, cudaStream_t st);
cudaError_t g_launch_ntt_inv(const GenCtx& c, const void* in, int64_t npoly, void* coef, cudaStream_t st);
cudaError_t g_launch_poly_mul(const GenCtx& c, const void* a, const void* b, int64_t npoly, void* out, cudaStream_t st);
cudaError_t g_launch_ref_repr(const GenCtx& c, const void* coef, int64_t npoly, void* out, cudaStream_t st);
cudaError_t g_launch_matvec(const GenCtx& c, const void* vec_coef, int64_t nvec, void* vec_ntt, void* y_ntt, void* y_coef,
                            cudaStream_t st);
cudaError_t g_launch_sign(const GenCtx& c, const void* sk_ntt, const void* ch_pairs, int ch_wt, int64_t n, void* sig,
                          cudaStream_t st);
cudaError_t g_launch_verify(const GenCtx& c, const void* vec_coef, const void* vk_ntt, const void* ch_pairs, int ch_wt,
                            const void* rhs_only, const void* extra_rhs, int64_t n, int64_t bd, int wt, uint8_t* verdict,
                            cudaStream_t st);
cudaError_t g_launch_vec_addsub(const GenCtx& c, const void* a, const void* b, int64_t nelem, int sub, void* out,
                                cudaStream_t st);
cudaError_t g_launch_agg_partial(const GenCtx& c, const void* sigs, const void* ag_pairs, int64_t count, void* partial,
                                 cudaStream_t st);
// general (non-monomial) aggregation coefficients: ag_pairs [count][ag_wt][2]
cudaError_t g_launch_agg_partial_poly(const GenCtx& c, const void* sigs, const void* ag_pairs, int ag_wt, int64_t count,
                                      void* partial, cudaStream_t st);
cudaError_t g_launch_aggv_partial_poly(const GenCtx& c, const void* vk_ntt, const void* ch_pairs, int ch_wt, const void* ag_pairs,
                                       int ag_wt, int64_t count, void* partial, cudaStream_t st);
cudaError_t g_launch_agg_finish(const GenCtx& c, const void* partial, void* ag_sig, cudaStream_t st);
cudaError_t g_launch_aggv_partial(const GenCtx& c, const void* vk_ntt, const void* ch_pairs, int ch_wt, const void* ag_pairs,
                                  int64_t count, void* partial, cudaStream_t st);
cudaError_t g_launch_aggv_finish(const GenCtx& c, const void* partial, const void* ag_sig, int64_t total, int64_t ag_cap,
                                 int64_t avf_bd, int avf_wt, uint8_t* verdict, cudaStream_t st);

struct RingCtx {
    ModQ m;
    StageConst sc;
    StageConstF scf;
    StageConstF iscf;          // warp-uniform twiddles of the FP32-assisted inverse (ntt_inv_256_fp), index half + j
    const NttTables* tab;      // device
    const uint32_t* a_hat;     // device, uint32[l][256]: NTT(key_ch), slot order
    int l;
    int num_sms;
};

cudaError_t launch_ntt_fwd(const RingCtx& c, const int16_t* coef, int64_t npoly, uint16_t* out, cudaStream_t st);
cudaError_t launch_ntt_ref_repr(const RingCtx& c, const int16_t* coef, int64_t npoly, int16_t* out, cudaStream_t st);
cudaError_t launch_ntt_inv(const RingCtx& c, const uint16_t* in, int64_t npoly, int16_t* coef, cudaStream_t st);
cudaError_t launch_poly_mul(const RingCtx& c, const int16_t* a, const int16_t* b, int64_t npoly, int16_t* out,
                            cudaStream_t st);
// y = key_ch * v for nvec coefficient-form vectors; optional v_ntt / y_coef outputs
cudaError_t launch_matvec(const RingCtx& c, const int16_t* vec_coef, int64_t nvec, uint16_t* vec_ntt,
                          uint16_t* y_ntt, int16_t* y_coef, cudaStream_t st);
cudaError_t launch_sign(const RingCtx& c, const uint16_t* sk_ntt, const int16_t* ch_pairs, int ch_wt, int64_t n,
                        int16_t* sig, cudaStream_t st);
// verdict = bounds(vec) && key_ch*vec == [vk_left*c] + [vk_right | rhs0] + [rhs1]
cudaError_t launch_verify(const RingCtx& c, const int16_t* vec_coef, const uint16_t* vk_ntt,
                          const int16_t* ch_pairs, int ch_wt, const uint16_t* rhs_only, const uint16_t* extra_rhs,
                          int64_t n, int bd, int wt, uint8_t* verdict, cudaStream_t st);
// the same on packed wire-format rows (sig_bits/vk_bits = 11/14 or 13/16); cudaErrorNotSupported otherwise.  st_packed
// (adaptor verify; nullable): statements packed at vk_bits bits, bias 0, 16-byte aligned at 16 bits
cudaError_t launch_verify_packed(const RingCtx& c, const uint8_t* sig_packed, int sig_bits, int sig_bias,
                                 const uint8_t* vk_packed, int vk_bits, const int16_t* ch_pairs, int ch_wt, int64_t n,
                                 int bd, int wt, uint8_t* verdict, cudaStream_t st, const uint8_t* st_packed = nullptr);
// sign straight into the wire format (sig_bits = 11 / 13, 16-byte aligned rows; cudaErrorNotSupported otherwise):
// sig_packed uint8[n][l][32*sig_bits], in_range (nullable) uint8[n][l], as launch_sign -> launch_pack would write them
cudaError_t launch_sign_packed(const RingCtx& c, const uint16_t* sk_ntt, const int16_t* ch_pairs, int ch_wt, int64_t n,
                               int sig_bits, int sig_bias, uint8_t* sig_packed, uint8_t* in_range, cudaStream_t st);
// sign from packed coefficient-form signing keys straight into the wire format (sign_sk.cu): sk_packed uint8[n][2][l][32*sk_bits]
// (bias sk_bias) -> sig_packed uint8[n][l][32*sig_bits], in_range (nullable) uint8[n][l], exactly as unpack -> launch_ntt_fwd ->
// launch_sign_packed would write them.  Rows of both packed buffers 16-byte aligned; cudaErrorNotSupported unless
// sign_sk_fused_applies.
inline bool sign_sk_fused_applies(int sk_bits, int sig_bits, int ch_bd, int ch_wt) {
    // bytes as fields (sk_bits <= 8), monomial challenges (ch_bd = 1): the 16-bit lane sums of the kernel stay below
    // ch_wt * 255 < 2^16 for every ch_wt <= d
    return (sk_bits == 7 || sk_bits == 8) && (sig_bits == 11 || sig_bits == 13) && ch_bd == 1 && ch_wt >= 1 && ch_wt <= D;
}
cudaError_t launch_sign_sk_packed(const RingCtx& c, const uint8_t* sk_packed, int sk_bits, int sk_bias,
                                  const int16_t* ch_pairs, int ch_bd, int ch_wt, int64_t n, int sig_bits, int sig_bias,
                                  uint8_t* sig_packed, uint8_t* in_range, cudaStream_t st);
cudaError_t launch_vec_addsub(const RingCtx& c, const int16_t* a, const int16_t* b, int64_t nelem, int sub,
                              int16_t* out, cudaStream_t st);
cudaError_t launch_agg_partial(const RingCtx& c, const int16_t* sigs, const int16_t* ag_pairs, int64_t count,
                               int32_t* partial, cudaStream_t st);
cudaError_t launch_agg_finish(const RingCtx& c, const int32_t* partial, int16_t* ag_sig, cudaStream_t st);
cudaError_t launch_aggv_partial(const RingCtx& c, const uint16_t* vk_ntt, const int16_t* ch_pairs, int ch_wt,
                                const int16_t* ag_pairs, int64_t count, int32_t* partial, cudaStream_t st);
cudaError_t launch_aggv_finish(const RingCtx& c, const int32_t* partial, const int16_t* ag_sig, int64_t total,
                               int ag_cap, int avf_bd, int avf_wt, uint8_t* verdict, cudaStream_t st);
// batches of aggregates (items sorted by group, gid from launch_group_ids): partial int32[n_agg][l][256] /
// int32[n_agg][256], zeroed by the caller; k_agg_finish over nelem elements; residues of the verify partials in [0, q);
// the lower limits k_verify does not check (1 <= count_g <= ag_cap, ag_sig != 0), ANDed into verdict.
// Packed inputs (wire format): signatures sig_bits = 11 / 13 (0 = int16), keys vk_bits = 14 (0 = uint16, which is also
// the 16-bit packing), aggregates 12 / 14 bits in the witness-verify form of k_verify; cudaErrorNotSupported otherwise
cudaError_t launch_agg_partial_seg(const RingCtx& c, const void* sigs, int sig_bits, int sig_bias, const int16_t* ag_pairs,
                                   const int32_t* gid, int64_t total, int64_t n_agg, int32_t* partial, cudaStream_t st);
cudaError_t launch_agg_finish_n(const RingCtx& c, const int32_t* partial, int64_t nelem, int16_t* ag_sig, cudaStream_t st);
cudaError_t launch_aggv_partial_seg(const RingCtx& c, const void* vk_ntt, int vk_bits, const int16_t* ch_pairs, int ch_wt,
                                    const int16_t* ag_pairs, const int32_t* gid, int64_t total, int64_t n_agg,
                                    int32_t* partial, cudaStream_t st);
cudaError_t launch_aggv_residues(const RingCtx& c, const int32_t* partial, int64_t nelem, uint16_t* out, cudaStream_t st);
cudaError_t launch_aggv_limits(const RingCtx& c, const int64_t* agg_off, int64_t n_agg, const int16_t* ag_sig, int64_t ag_cap,
                               uint8_t* verdict, cudaStream_t st);
cudaError_t launch_aggv_limits_packed(const RingCtx& c, const int64_t* agg_off, int64_t n_agg, const uint8_t* ag_packed, int bits,
                                      int bias, int64_t ag_cap, uint8_t* verdict, cudaStream_t st);
// witness-verify form of k_verify on packed rows (bias `bias`): (bits, rhs_bits) = (12 | 14, 16), (2, 16), (2 | 12, 14); a
// 14-bit rhs_only is a packed row uint8[n][32*14] (bias 0).  cudaErrorNotSupported otherwise.
cudaError_t launch_verify_rhs_packed(const RingCtx& c, const uint8_t* vec_packed, int bits, int bias, const uint16_t* rhs_only,
                                     int64_t n, int bd, int wt, uint8_t* verdict, cudaStream_t st, int rhs_bits = 16);

// wire format (wire.cu): `bits`-bit little-endian packing of (x + bias) mod 2^16, 32*bits bytes per polynomial
cudaError_t launch_pack(const RingCtx& c, const void* in, int64_t npoly, int bits, int bias, uint8_t* out,
                        uint8_t* in_range, cudaStream_t st);
cudaError_t launch_unpack(const RingCtx& c, const uint8_t* in, int64_t npoly, int bits, int bias, void* out,
                          cudaStream_t st);
// unpack both operands -> k_vec_addsub (a + b, or a - b when sub) -> k_pack in one pass, any widths 1..16 (adaptor adapt /
// extract on the wire format): a, b, out uint8[npoly][32*bits of each], in_range (nullable) uint8[npoly]
cudaError_t launch_addsub_packed(const RingCtx& c, const uint8_t* a, int a_bits, int a_bias, const uint8_t* b, int b_bits,
                                 int b_bias, int sub, int64_t npoly, int bits, int bias, uint8_t* out, uint8_t* in_range,
                                 cudaStream_t st);
// k_agg_finish + k_pack in one pass: BKLM partial sums int32[npoly][256] -> packed aggregates and in_range flags
cudaError_t launch_agg_finish_pack(const RingCtx& c, const int32_t* partial, int64_t npoly, int bits, int bias, uint8_t* out,
                                   uint8_t* in_range, cudaStream_t st);

// content-mode hash inputs (content.cu).  coef int16[n][rows][256] (rows 1 or 2) -> out uint8[n][57]: '<' + name + ' ' +
// SHAKE256(prefix || rows).hexdigest(16) + '>'; prefix = name || le16(secpar) (24 bytes), head = '<' + name + ' '
cudaError_t launch_content_str(const RingCtx& c, const int16_t* coef, int64_t n, int rows, const uint8_t (&prefix)[24],
                               const uint8_t (&head)[24], uint8_t* out, cudaStream_t st);
// out / out_off (lcb_challenge_inputs_batch); msg_i = msg[msg_off[i] - shift .. msg_off[i+1] - shift); out_len bytes of out
cudaError_t launch_challenge_inputs(const RingCtx& c, const uint8_t* st_str, const uint8_t* vk_str, const uint8_t* msg,
                                    int64_t shift, const int64_t* msg_off, int64_t n, int64_t out_len, uint8_t* out,
                                    int64_t* out_off, cudaStream_t st);
// agmsg of lcb_aggregation_inputs_batch at the group offsets ag_off[n_agg+1] the caller computed; gid from launch_group_ids
cudaError_t launch_aggregation_inputs(const RingCtx& c, const int64_t* agg_off, const int64_t* ag_off, int64_t n_agg,
                                      const int32_t* gid, int64_t total, const uint8_t* vk_str, const uint8_t* msg,
                                      int64_t shift, const int64_t* msg_off, int64_t out_len, uint8_t* out, cudaStream_t st);

}  // namespace lcb
