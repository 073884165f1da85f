/* lcb200 — C ABI of the B200-native batched engine for the lattice-cryptography hot path.
 *
 * The reference (b-g-goodell/lattice-cryptography) is pure Python and has no FFI; its seam is
 * the ten names it imports from `lattice_algebra` (one_time_keys.py:4-5, lm_one_time_sigs.py:3,
 * bklm_one_time_agg_sigs.py:1, adaptor_sigs.py:1) plus its scheme functions.  Each entry point
 * below names the reference code it replaces.  See INTEGRATION.md for the ctypes binding.
 *
 * Conventions
 *   - every function returns 0 (LCB_OK) or a negative lcb_status; nothing throws across the ABI;
 *   - the caller owns every buffer; a data pointer may be HOST or DEVICE memory (detected per
 *     call with cudaPointerGetAttributes; host buffers are staged through engine-owned device
 *     scratch inside the call); scalar/offset arrays follow the same rule;
 *   - one ctx = one GPU + one ordered stream; a ctx is not re-entrant; distinct ctxs are independent;
 *   - calls are asynchronous only when EVERY buffer is device memory; otherwise they return after
 *     the results are in the caller's host buffer.  lcb_synchronize() waits for the stream.
 *
 * Data formats (d = ring degree, a power of two in 32..1024; l = vector length; q prime, q = 1 mod 2d)
 *   coefficient form : int16_t[d], centred residues in [-(q-1)/2, (q-1)/2], natural order
 *   NTT form         : uint16_t[d], residues in [0, q); slot p holds a(psi^(2*bitrev_logd(p)+1)),
 *                      psi = least primitive 2d-th root of unity mod q (the reference's `rou`)
 *   pairs            : int16_t[wt][2] = (index, coefficient) in sampler DRAW ORDER
 *   ragged bytes     : uint8_t blob + int64_t off[n+1]; item i is blob[off[i] .. off[i+1])
 * WIDE contexts (q >= 2^16, up to 2^31): every int16_t / uint16_t array of this header then holds int32_t /
 * uint32_t elements of the same shape, and the int32_t BKLM partial sums become int64_t; pass the wider arrays
 * through the same pointers.  The shipped parameter sets (d = 256, q = 11777 / 39937) run on register-resident
 * half-warp kernels; every other (d, q) runs on one-polynomial-per-warp shared-memory kernels (ring_generic.cu).
 * Caller-owned DEVICE buffers of 16-bit data must be 16-byte aligned (LCB_ERR_CUDA, "misaligned address", otherwise).
 */
#ifndef LCB200_H
#define LCB200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct lcb_ctx lcb_ctx;

typedef enum lcb_status {
    LCB_OK = 0,
    LCB_ERR_INVALID = -1,      /* bad argument / unsupported parameter set            */
    LCB_ERR_CUDA = -2,         /* a CUDA runtime call failed (see lcb_last_error)     */
    LCB_ERR_NO_DEVICE = -3,    /* no sm_100 device; there is NO CPU fallback          */
    LCB_ERR_NO_KEY_CH = -4,    /* an operation needs key_ch and lcb_set_key_ch was not called */
    LCB_ERR_OOM = -5
} lcb_status;

#define LCB_SALT_MAX 32

/* Scheme constants, mirroring the reference's `pp` dict (lm_one_time_sigs.py:36-55,
 * bklm_one_time_agg_sigs.py:27-44, adaptor_sigs.py:37-71).  Salts are NUL-terminated ASCII. */
typedef struct lcb_scheme {
    int32_t sk_bd, sk_wt;
    int32_t ch_bd, ch_wt;
    int32_t ag_bd, ag_wt;
    int32_t wit_bd, wit_wt;
    char sk_salt[LCB_SALT_MAX];   /* 'SK_SALT' (the engine appends LEFT / RIGHT)           */
    char ch_salt[LCB_SALT_MAX];   /* 'CH_SALT'                                             */
    char ag_salt[LCB_SALT_MAX];   /* 'AG_SALT' (the engine appends the decimal index)      */
    char wit_salt[LCB_SALT_MAX];  /* 'WIT_SALT'                                            */
} lcb_scheme;

const char* lcb_strerror(int status);
const char* lcb_last_error(const lcb_ctx* ctx);     /* detail string of the last failure    */
int lcb_version(void);
/* 1 for the checked build (make CHECKED=1: device-side asserts on every hand-rolled bound of a global access - the
 * stand-in for compute-sanitizer's memcheck, which is not available on the GPU pool), 0 for the production build.
 * lcb_checked_selftest launches a kernel whose check fails on purpose: LCB_OK on the production build, LCB_ERR_CUDA
 * ("device-side assert triggered", the context is unusable afterwards) on the checked one - proof that checks are live. */
int lcb_build_is_checked(void);
int lcb_checked_selftest(lcb_ctx* ctx);

/* LatticeParameters(modulus=q, degree=d, length=l) + secpar (lattice_algebra; constructed at
 * lm_one_time_sigs.py:19-21; the reference's container tests use (d, q) = (32, 193), tests/test_one_time_keys.py:12-33).
 * Supported: d a power of two in 32..1024, 3 <= q < 2^31 prime with q % (2d) == 1, 1 <= l <= 64,
 * 1 <= secpar <= 512.  device = CUDA ordinal. */
int lcb_ctx_create(lcb_ctx** out, int device, int secpar, int q, int d, int l);
int lcb_ctx_destroy(lcb_ctx* ctx);
int lcb_ctx_set_stream(lcb_ctx* ctx, void* cuda_stream);   /* run on a caller-owned cudaStream_t  */
int lcb_synchronize(lcb_ctx* ctx);
int lcb_ctx_root_of_unity(const lcb_ctx* ctx);             /* == LatticeParameters.rou            */

/* SchemeParameters.key_ch (one_time_keys.py:259-299): upload the public row, coefficient form
 * int16[l][d]; kept NTT-resident on the device until replaced. */
int lcb_set_key_ch(lcb_ctx* ctx, const int16_t* key_ch_coef);

/* hashlib.shake_256(item).digest(out_len) per item (lattice_algebra binary_digest without salt). */
int lcb_shake256_batch(lcb_ctx* ctx, const uint8_t* in, const int64_t* in_off, int64_t n,
                       uint8_t* out, int64_t out_len);

/* The unseeded keygen path for batches (make_random_seed, lm_one_time_sigs.py:58-61, draws secpar random bits per
 * key from the OS): ONE 32-byte secret from the host's entropy source is expanded on the device into n seed
 * bitstrings, seed i = the first secpar bits (most significant bit of each byte first) of
 * SHAKE256(secret32 || le64(first + i)) as ASCII '0'/'1' - exactly the strings keygen hashes, so seed i reproduces
 * key i.  seeds: uint8[n][secpar] (host or device); feed it to lcb_lm_keygen_batch with seed_off[i] = i * secpar. */
int lcb_expand_seeds(lcb_ctx* ctx, const uint8_t* secret32, int64_t first, int64_t n, uint8_t* seeds);

/* hash2polynomialvector / hash2polynomial (lm_one_time_sigs.py:70-91,142-160;
 * adaptor_sigs.py:86-96): SHAKE256(salt || item_i) -> vec_len polynomials with `wt` distinct
 * non-zero positions and coefficients in +-[1..bd].  Either output may be NULL.
 *   out_dense : int16[n][vec_len][d]    out_pairs : int16[n][vec_len][wt][2] */
int lcb_hash2polyvec_batch(lcb_ctx* ctx, const char* salt, const uint8_t* msgs, const int64_t* msg_off,
                           int64_t n, int bd, int wt, int vec_len, int16_t* out_dense, int16_t* out_pairs);

/* Polynomial.__init__ / get_coef_rep / __mul__ (lattice_algebra): transforms and the negacyclic
 * product, npoly independent polynomials. */
int lcb_ntt_fwd_batch(lcb_ctx* ctx, const int16_t* coef, int64_t npoly, uint16_t* ntt);
int lcb_ntt_inv_batch(lcb_ctx* ctx, const uint16_t* ntt, int64_t npoly, int16_t* coef);
int lcb_poly_mul_batch(lcb_ctx* ctx, const int16_t* a, const int16_t* b, int64_t npoly, int16_t* out);
/* Polynomial.ntt_representation exactly as lattice_algebra stores it (parity level L3): the 2d-point
 * cyclic transform of the zero-padded coefficients, natural order, centred: rep[k] = a(rou^k), int16[npoly][2d]. */
int lcb_ntt_reference_repr_batch(lcb_ctx* ctx, const int16_t* coef, int64_t npoly, int16_t* rep);

/* make_one_key / keygen_core (lm_one_time_sigs.py:64-97,126-138; adaptor_sigs.py:104-137).
 * seeds: ragged ASCII bitstrings.  Any output may be NULL.
 *   sk_coef int16[n][2][l][d], sk_ntt uint16[n][2][l][d], vk_ntt uint16[n][2][d], vk_coef int16[n][2][d] */
int lcb_lm_keygen_batch(lcb_ctx* ctx, const lcb_scheme* sch, const uint8_t* seeds, const int64_t* seed_off,
                        int64_t n, int16_t* sk_coef, uint16_t* sk_ntt, uint16_t* vk_ntt, int16_t* vk_coef);

/* make_signature_challenge (lm_one_time_sigs.py:141-160; adaptor_sigs.py:168-188): chmsg item i is
 * the full hash input after the salt, i.e. str(otvk)+', '+msg.  out_pairs int16[n][ch_wt][2]. */
int lcb_challenge_batch(lcb_ctx* ctx, const lcb_scheme* sch, const uint8_t* chmsg, const int64_t* chmsg_off,
                        int64_t n, int16_t* out_pairs);

/* sign (lm_one_time_sigs.py:163-170) and adaptor presign (adaptor_sigs.py:191-195):
 * sig = sk_left ** c + sk_right, sig int16[n][l][d] coefficient form. */
int lcb_lm_sign_batch(lcb_ctx* ctx, const lcb_scheme* sch, const uint16_t* sk_ntt, const uint8_t* chmsg,
                      const int64_t* chmsg_off, int64_t n, int16_t* sig);

/* verify (lm_one_time_sigs.py:173-191), adaptor preverify / verify (adaptor_sigs.py:198-217,247-266):
 * verdict[i] = max|sig_i| <= bd && max weight <= wt && key_ch*sig == vk_left*c + vk_right (+ st).
 * st_ntt may be NULL (LM verify, preverify) or uint16[n][d] (adaptor verify).
 * The bound is tested on the int16 values AS GIVEN: coefficient-form inputs MUST be centred residues (what every
 * engine entry point emits and what the reference's get_coef_rep() returns).  A non-canonical representative
 * such as x + q is not re-centred first; it fails the bound (verdict 0) whenever |x + q| > bd.
 * At most 2^30 items per call (LCB_ERR_INVALID beyond; the same for the packed and the witness-verify entry points). */
int lcb_lm_verify_batch(lcb_ctx* ctx, const lcb_scheme* sch, const uint16_t* vk_ntt, const uint8_t* chmsg,
                        const int64_t* chmsg_off, const int16_t* sig, const uint16_t* st_ntt, int64_t n,
                        int bd, int wt, uint8_t* verdict);

/* ---- Packed wire format (SURVEY.md 8(f)2).  The reference has no serialisation: keys print as memory
 * addresses and signatures are live Python objects (one_time_keys.py:197-237), so this format is the
 * engine's own and opt-in.  A polynomial is its 256 values v_i = (x_i + bias) mod 2^16, `bits` bits each,
 * value i at bit offset i*bits, least significant bit first: 32*bits bytes per polynomial, polynomials
 * back to back.  Signatures: x = centred coefficient, bias = vf_bd, bits = ceil(log2(2*vf_bd+1)) (11 at
 * secpar 128, 13 at 256).  NTT-form keys: x = slot value, bias = 0, bits = ceil(log2 q) (14 / 16).
 * Defined for d == 256, q < 2^16 contexts (LCB_ERR_INVALID otherwise).
 * `values` is int16 or uint16 [npoly][d]; packed buffers must be 4-byte aligned (LCB_ERR_INVALID otherwise);
 * lcb_lm_verify_packed_batch reads the shipped widths directly only from 16-byte aligned device buffers and
 * unpacks into scratch first when a caller-owned device buffer is merely 4-byte aligned.
 * in_range (nullable) uint8[npoly]: 1 when every value of the polynomial was representable. */
int lcb_pack_batch(lcb_ctx* ctx, const void* values, int64_t npoly, int bits, int bias, uint8_t* packed,
                   uint8_t* in_range);
int lcb_unpack_batch(lcb_ctx* ctx, const uint8_t* packed, int64_t npoly, int bits, int bias, void* values);

/* lcb_lm_verify_batch (verify, lm_one_time_sigs.py:173-191) on packed inputs: vk_packed uint8[n][2][32*vk_bits]
 * (bias 0), sig_packed uint8[n][l][32*sig_bits] (bias sig_bias).  Same verdicts as unpacking first.  The shipped
 * widths (sig/vk = 11/14 and 13/16 bits) are read by the verify kernel directly; other widths are unpacked
 * into engine scratch first.  Host-resident signatures (here and in lcb_lm_verify_batch) cross PCIe in
 * chunks on a second stream while the kernels of the previous chunk run. */
int lcb_lm_verify_packed_batch(lcb_ctx* ctx, const lcb_scheme* sch, const uint8_t* vk_packed, int vk_bits,
                               const uint8_t* chmsg, const int64_t* chmsg_off, const uint8_t* sig_packed,
                               int sig_bits, int sig_bias, int64_t n, int bd, int wt, uint8_t* verdict);

/* ---- The other records that leave a signer, on the packed wire format.  Same rules as the packed calls above: bits
 * 1..16, biases 0..32767, packed buffers 4-byte aligned (LCB_ERR_INVALID otherwise); d == 256, q < 2^16 contexts only
 * (LCB_ERR_INVALID, "the packed wire format is defined for d == 256, q < 2^16 contexts only"); host or device buffers
 * with the usual synchronisation rules.  Each result is exactly that of the composition named, for any input bytes.
 * Shipped packings: presignatures in ceil(log2(2 pvf_bd + 1)) bits with bias pvf_bd (11 / 13 bits), adaptor signatures
 * with vf_bd (11 / 13), statements like keys (14 / 16 bits, bias 0).  Signatures made from genuine keys lie within
 * sk_bd (1 + ch_wt) = vf_bd, so their in_range flags are 1. */

/* sign (lm_one_time_sigs.py:163-170) / adaptor presign (adaptor_sigs.py:191-195) into packed rows:
 * sig_packed uint8[n][l][32*sig_bits] (bias sig_bias), in_range (nullable) uint8[n][l].
 * Exactly lcb_lm_sign_batch -> lcb_pack_batch(sig_bits, sig_bias), for any sk_ntt values.  11- and 13-bit rows in
 * 16-byte aligned buffers are written by the sign kernel itself; other widths sign into engine scratch and pack. */
int lcb_lm_sign_packed_batch(lcb_ctx* ctx, const lcb_scheme* sch, const uint16_t* sk_ntt, const uint8_t* chmsg,
                             const int64_t* chmsg_off, int64_t n, int sig_bits, int sig_bias,
                             uint8_t* sig_packed, uint8_t* in_range);

/* ---- Keys on the packed wire format.  A packed signing key is uint8[2][l][32*sk_bits]: the rows of sk_left, then those of
 * sk_right, each a COEFFICIENT-form polynomial packed as above (x = centred coefficient, bias sk_bias).  Shipped packing:
 * sk_bits = ceil(log2(2 sk_bd + 1)) with bias sk_bd - 7 bits / bias 45 at secpar 128, 8 bits / bias 65 at 256: 224 / 256
 * bytes per row, 5,824 / 11,776 bytes per key instead of 13,312 / 23,552 for the uint16 NTT form.  Verification keys keep
 * their packing (NTT form, 14 / 16 bits, bias 0).  Same rules as the packed calls above (bits 1..16, biases 0..32767, packed
 * buffers 4-byte aligned, d == 256 and q < 2^16 only, host or device buffers), at most 2^30 items.  Signing keys are secret:
 * host-resident ones are staged through engine scratch that is cleared afterwards. */

/* keygen (lm_one_time_sigs.py:64-97,126-138) into packed keys: exactly lcb_lm_keygen_batch(sk_coef, vk_ntt) ->
 * lcb_pack_batch(sk_coef, sk_bits, sk_bias, sk_in_range) and lcb_pack_batch(vk_ntt, vk_bits, 0).  sk_packed
 * uint8[n][2][l][32*sk_bits], sk_in_range uint8[n][2][l], vk_packed uint8[n][2][32*vk_bits]; each may be NULL, but not both
 * sk_packed and vk_packed.  The 16-bit keys stay in engine scratch, chunk by chunk.  Needs key_ch (LCB_ERR_NO_KEY_CH). */
int lcb_lm_keygen_packed_batch(lcb_ctx* ctx, const lcb_scheme* sch, const uint8_t* seeds, const int64_t* seed_off, int64_t n,
                               int sk_bits, int sk_bias, uint8_t* sk_packed, uint8_t* sk_in_range, int vk_bits,
                               uint8_t* vk_packed);

/* sign (lm_one_time_sigs.py:163-170) / adaptor presign (adaptor_sigs.py:191-195) from packed signing keys into packed rows:
 * exactly lcb_unpack_batch(sk_packed, 2 n l, sk_bits, sk_bias) -> lcb_ntt_fwd_batch -> lcb_lm_sign_packed_batch(sig_bits,
 * sig_bias), for any bytes in sk_packed.  sig_packed uint8[n][l][32*sig_bits], in_range (nullable) uint8[n][l].  7- and 8-bit
 * keys with 11- and 13-bit signatures, monomial challenges (ch_bd == 1) and 16-byte aligned buffers are signed by one kernel
 * that sums the rotations of the packed rows; anything else is unpacked and transformed into engine scratch first. */
int lcb_lm_sign_packed_sk_batch(lcb_ctx* ctx, const lcb_scheme* sch, const uint8_t* sk_packed, int sk_bits, int sk_bias,
                                const uint8_t* chmsg, const int64_t* chmsg_off, int64_t n, int sig_bits, int sig_bias,
                                uint8_t* sig_packed, uint8_t* in_range);

/* adaptor verify (adaptor_sigs.py:247-266) from packed keys (bias 0), signatures (bias sig_bias) and statements
 * st_packed uint8[n][32*st_bits] (NTT form, bias 0, packed like a key half).  Exactly unpack all three ->
 * lcb_lm_verify_batch(st_ntt = the unpacked statements).  st_packed must not be NULL (preverify is
 * lcb_lm_verify_packed_batch with bd = pvf_bd).  At most 2^30 items.  The shipped widths with st_bits == vk_bits are
 * read by the verify kernel directly (16-bit key and statement rows from 16-byte aligned buffers); anything else is
 * unpacked into engine scratch first. */
int lcb_adaptor_verify_packed_batch(lcb_ctx* ctx, const lcb_scheme* sch, const uint8_t* vk_packed, int vk_bits,
                                    const uint8_t* chmsg, const int64_t* chmsg_off, const uint8_t* sig_packed,
                                    int sig_bits, int sig_bias, const uint8_t* st_packed, int st_bits,
                                    int64_t n, int bd, int wt, uint8_t* verdict);

/* adapt (adaptor_sigs.py:220-221): exactly unpack(presig) -> lcb_vec_add_batch(presig, wit) -> lcb_pack_batch.
 * presig_packed uint8[npoly][32*presig_bits], wit_coef int16[npoly][d], sig_packed uint8[npoly][32*sig_bits],
 * in_range (nullable) uint8[npoly]. */
int lcb_adaptor_adapt_packed_batch(lcb_ctx* ctx, const uint8_t* presig_packed, int presig_bits, int presig_bias,
                                   const int16_t* wit_coef, int64_t npoly, int sig_bits, int sig_bias,
                                   uint8_t* sig_packed, uint8_t* in_range);

/* extract (adaptor_sigs.py:224-226): exactly unpack both -> lcb_vec_sub_batch(sig, presig); wit_coef int16[npoly][d]. */
int lcb_adaptor_extract_packed_batch(lcb_ctx* ctx, const uint8_t* sig_packed, int sig_bits, int sig_bias,
                                     const uint8_t* presig_packed, int presig_bits, int presig_bias, int64_t npoly,
                                     int16_t* wit_coef);

/* make_agg_coefs (bklm_one_time_agg_sigs.py:78-81): coefficient i = H2P(ag_salt+str(first+i) || agmsg),
 * out_pairs int16[count][ag_wt][2].  ag_wt = ag_bd = 1 (the shipped tables: signed monomials) takes the dedicated
 * shared-message kernels; any other 1 <= ag_wt <= d, ag_bd >= 1 runs the full sampler per coefficient. */
int lcb_bklm_agg_coefs(lcb_ctx* ctx, const lcb_scheme* sch, const uint8_t* agmsg, int64_t agmsg_len,
                       int64_t first, int64_t count, int16_t* out_pairs);

/* aggregate (bklm_one_time_agg_sigs.py:92-96), one shard: partial[l][d] (int32, residues mod q,
 * not centred; ag_pairs int16[count][ag_wt][2], general polynomials when ag_wt > 1 or ag_bd > 1)
 * = sum_i sig_sorted[i] ** ag_i over this shard's `count` signatures whose global
 * sorted positions start at `first`.  ag_pairs from lcb_bklm_agg_coefs (same first/count) or NULL to
 * derive them here from agmsg.  Shards are summed by the caller (NCCL reduce) and finished below. */
int lcb_bklm_aggregate_partial(lcb_ctx* ctx, const lcb_scheme* sch, const int16_t* sig_sorted,
                               const int16_t* ag_pairs, const uint8_t* agmsg, int64_t agmsg_len,
                               int64_t first, int64_t count, int32_t* partial);
int lcb_bklm_aggregate_finish(lcb_ctx* ctx, const int32_t* partial_sum, int16_t* ag_sig);

/* aggregate_verify (bklm_one_time_agg_sigs.py:99-116), one shard of the right-hand side:
 * partial[d] (int32 mod q, NTT form) = sum_i (vk_left_i*c_i + vk_right_i) * ag_i. */
int lcb_bklm_aggverify_partial(lcb_ctx* ctx, const lcb_scheme* sch, const uint16_t* vk_ntt_sorted,
                               const uint8_t* chmsg_sorted, const int64_t* chmsg_off, const int16_t* ag_pairs,
                               const uint8_t* agmsg, int64_t agmsg_len, int64_t first, int64_t count,
                               int32_t* partial);
/* bounds 1 <= n <= avf_bd, 1 <= w <= avf_wt, 1 <= total <= ag_cap, then key_ch*ag_sig == sum. */
int lcb_bklm_aggverify_finish(lcb_ctx* ctx, const int32_t* partial_sum, const int16_t* ag_sig, int64_t total,
                              int ag_cap, int avf_bd, int avf_wt, uint8_t* verdict);

/* ---- Batches of independent aggregates: many small aggregates (the reference caps one at ag_cap = 2 signatures) in one
 * call instead of a handful of launches, copies and synchronisations per aggregate.  Whole aggregates only: a group is
 * never split across calls (the shard entry points above do that).  Group g covers sorted items
 * [agg_off[g], agg_off[g+1]); offset arrays have n_agg + 1 entries.  Host-resident offset arrays must start at 0 and
 * never decrease (LCB_ERR_INVALID otherwise); device-resident ones are trusted.  The call reads agg_off[n_agg] and
 * agmsg_off[n_agg] on the host (a device array costs one small copy and a synchronisation).  At most 2^30 signatures
 * and 2^30 aggregates per call; n_agg == 0 returns LCB_OK.
 * The shipped geometry (d = 256, q < 2^16) with ag_wt = ag_bd = 1 runs segmented kernels over the whole batch; generic
 * contexts and non-monomial coefficients loop over the groups through the single-aggregate kernels: correct, not fast. */

/* aggregate (bklm_one_time_agg_sigs.py:92-96) for n_agg independent aggregates in one call.
 * Aggregate g covers the SORTED signatures [agg_off[g], agg_off[g+1]) of sig_sorted int16[agg_off[n_agg]][l][d];
 * its coefficients are H2P(ag_salt + str(j) || agmsg_g) for j = 0 .. count_g - 1 (the index restarts in every
 * aggregate), agmsg_g = agmsg[agmsg_off[g] .. agmsg_off[g+1]).  ag_sig int16[n_agg][l][d].
 * Every aggregate must hold >= 1 signature (LCB_ERR_INVALID otherwise); at most 2^30 signatures per call. */
int lcb_bklm_aggregate_batch(lcb_ctx* ctx, const lcb_scheme* sch, const int64_t* agg_off, int64_t n_agg,
                             const int16_t* sig_sorted, const uint8_t* agmsg, const int64_t* agmsg_off,
                             int16_t* ag_sig);

/* aggregate_verify (:99-116) for n_agg aggregates.  vk_ntt_sorted uint16[total][2][d], chmsg_sorted ragged over the
 * same total items, ag_sig int16[n_agg][l][d], verdict uint8[n_agg].  verdict[g] is exactly what
 * lcb_bklm_aggverify_partial(first = 0, count_g) + lcb_bklm_aggverify_finish(total = count_g) give for that group;
 * an empty group, or one above ag_cap, gets verdict 0 (not an error). */
int lcb_bklm_aggregate_verify_batch(lcb_ctx* ctx, const lcb_scheme* sch, const int64_t* agg_off, int64_t n_agg,
                                    const uint16_t* vk_ntt_sorted, const uint8_t* chmsg_sorted,
                                    const int64_t* chmsg_off, const uint8_t* agmsg, const int64_t* agmsg_off,
                                    const int16_t* ag_sig, int ag_cap, int avf_bd, int avf_wt, uint8_t* verdict);

/* The same two calls on the packed wire format (d = 256, q < 2^16 only; LCB_ERR_INVALID with "the packed wire format is
 * defined for d == 256, q < 2^16 contexts only" otherwise).  An aggregate is packed like a signature, in
 * ceil(log2(2 avf_bd + 1)) bits with bias avf_bd (12 bits at secpar 128, 14 at 256).  Results are exactly those of
 * lcb_unpack_batch -> the unpacked batch call -> lcb_pack_batch, for any bytes in the packed buffers.  bits 1..16,
 * biases 0..32767, packed buffers 4-byte aligned (LCB_ERR_INVALID otherwise); the other checks and limits are those of
 * the unpacked calls.  Monomial coefficients with the shipped widths (signatures 11 / 13, keys 14 / 16, aggregates 12 / 14
 * bits) and 16-byte aligned rows are read and written by the kernels directly; anything else is unpacked into scratch
 * first.
 * aggregate (bklm_one_time_agg_sigs.py:92-96): sig_packed uint8[agg_off[n_agg]][l][32*sig_bits] (bias sig_bias) ->
 * ag_packed uint8[n_agg][l][32*ag_bits] (bias ag_bias) and in_range (nullable) uint8[n_agg][l], as lcb_pack_batch sets it. */
int lcb_bklm_aggregate_packed_batch(lcb_ctx* ctx, const lcb_scheme* sch, const int64_t* agg_off, int64_t n_agg,
                                    const uint8_t* sig_packed, int sig_bits, int sig_bias,
                                    const uint8_t* agmsg, const int64_t* agmsg_off,
                                    int ag_bits, int ag_bias, uint8_t* ag_packed, uint8_t* in_range);
/* aggregate_verify (:99-116) from packed keys uint8[total][2][32*vk_bits] (bias 0) and packed aggregates
 * uint8[n_agg][l][32*ag_bits] (bias ag_bias); verdict uint8[n_agg].  A key slot v >= q (possible at 14 and 16 bits) acts
 * as v mod q, here and in lcb_bklm_aggregate_verify_batch. */
int lcb_bklm_aggregate_verify_packed_batch(lcb_ctx* ctx, const lcb_scheme* sch, const int64_t* agg_off, int64_t n_agg,
                                           const uint8_t* vk_packed, int vk_bits,
                                           const uint8_t* chmsg_sorted, const int64_t* chmsg_off,
                                           const uint8_t* agmsg, const int64_t* agmsg_off,
                                           const uint8_t* ag_packed, int ag_bits, int ag_bias,
                                           int ag_cap, int avf_bd, int avf_wt, uint8_t* verdict);

/* adaptor make_one_wit / witgen (adaptor_sigs.py:80-101,140-151):
 *   wit_coef int16[n][l][d], st_ntt uint16[n][d], st_coef int16[n][d]; any may be NULL. */
int lcb_adaptor_witgen_batch(lcb_ctx* ctx, const lcb_scheme* sch, const uint8_t* seeds, const int64_t* seed_off,
                             int64_t n, int16_t* wit_coef, uint16_t* st_ntt, int16_t* st_coef);
/* adapt = presig + wit (adaptor_sigs.py:220-221); extract = sig - presig (:224-226); int16[n][l][d]. */
int lcb_vec_add_batch(lcb_ctx* ctx, const int16_t* a, const int16_t* b, int64_t npoly, int16_t* out);
int lcb_vec_sub_batch(lcb_ctx* ctx, const int16_t* a, const int16_t* b, int64_t npoly, int16_t* out);
/* witness_verify (adaptor_sigs.py:229-237): bounds + key_ch*wit == st. */
int lcb_adaptor_witness_verify_batch(lcb_ctx* ctx, const int16_t* wit_coef, const uint16_t* st_ntt, int64_t n,
                                     int bd, int wt, uint8_t* verdict);

/* ---- Adaptor witnesses on the packed wire format.  A packed witness is uint8[l][32*wit_bits]: coefficient-form rows packed
 * like a signature (x = centred coefficient, bias wit_bias).  Shipped packings: generated witnesses in
 * ceil(log2(2 wit_bd + 1)) = 2 bits with bias wit_bd = 1 (832 / 1,472 bytes per witness at secpar 128 / 256 instead of
 * 6,656 / 11,776 as int16); extracted witnesses in ceil(log2(2 ext_wit_bd + 1)) bits with bias ext_wit_bd (12 / 14 bits),
 * lossless for every witness witness_verify can accept.  Statements are packed like key halves (NTT form, bias 0, 14 / 16
 * bits).  Same rules as the packed calls above (bits 1..16, biases 0..32767, packed buffers 4-byte aligned, d == 256 and
 * q < 2^16 only, host or device buffers).  Each result is exactly that of the composition named, for any input bytes.
 * Witnesses are secret: host-resident ones are staged through engine scratch that is cleared afterwards. */

/* witgen (adaptor_sigs.py:80-101,140-151) into packed records: exactly lcb_adaptor_witgen_batch(wit_coef, st_ntt) ->
 * lcb_pack_batch(wit_coef, wit_bits, wit_bias, wit_in_range) and lcb_pack_batch(st_ntt, st_bits, 0).  wit_packed
 * uint8[n][l][32*wit_bits], wit_in_range uint8[n][l], st_packed uint8[n][32*st_bits]; each may be NULL, but not both
 * wit_packed and st_packed.  The 16-bit witnesses stay in engine scratch, chunk by chunk.  Needs key_ch
 * (LCB_ERR_NO_KEY_CH); at most 2^30 items. */
int lcb_adaptor_witgen_packed_batch(lcb_ctx* ctx, const lcb_scheme* sch, const uint8_t* seeds, const int64_t* seed_off,
                                    int64_t n, int wit_bits, int wit_bias, uint8_t* wit_packed, uint8_t* wit_in_range,
                                    int st_bits, uint8_t* st_packed);

/* witness_verify (adaptor_sigs.py:229-237) on packed witnesses and statements: exactly lcb_unpack_batch of both (statements
 * with bias 0, as uint16) -> lcb_adaptor_witness_verify_batch.  Needs key_ch; at most 2^30 items.  Witness / statement
 * widths 2 / 14 and 12 / 14 (secpar 128), 2 / 16 and 14 / 16 (secpar 256), with statements at the key width ceil(log2 q),
 * 16-byte aligned witness rows and 16-bit statement rows, are read by the verify kernel directly; anything else is
 * unpacked into engine scratch first. */
int lcb_adaptor_witness_verify_packed_batch(lcb_ctx* ctx, const uint8_t* wit_packed, int wit_bits, int wit_bias,
                                            const uint8_t* st_packed, int st_bits, int64_t n, int bd, int wt,
                                            uint8_t* verdict);

/* adapt (adaptor_sigs.py:220-221) with a packed witness: exactly unpack both -> lcb_vec_add_batch(presig, wit) ->
 * lcb_pack_batch(sig_bits, sig_bias, in_range).  presig_packed uint8[npoly][32*presig_bits], wit_packed
 * uint8[npoly][32*wit_bits], sig_packed uint8[npoly][32*sig_bits], in_range (nullable) uint8[npoly].  One kernel pass at
 * every width. */
int lcb_adaptor_adapt_packed_wit_batch(lcb_ctx* ctx, const uint8_t* presig_packed, int presig_bits, int presig_bias,
                                       const uint8_t* wit_packed, int wit_bits, int wit_bias, int64_t npoly, int sig_bits,
                                       int sig_bias, uint8_t* sig_packed, uint8_t* in_range);

/* extract (adaptor_sigs.py:224-226) into packed witnesses: exactly unpack both -> lcb_vec_sub_batch(sig, presig) ->
 * lcb_pack_batch(wit_bits, wit_bias, in_range).  wit_packed uint8[npoly][32*wit_bits], in_range (nullable) uint8[npoly].
 * At 2 bits a valid witness that is not the genuine one does not fit: in_range says so. */
int lcb_adaptor_extract_packed_wit_batch(lcb_ctx* ctx, const uint8_t* sig_packed, int sig_bits, int sig_bias,
                                         const uint8_t* presig_packed, int presig_bits, int presig_bias, int64_t npoly,
                                         int wit_bits, int wit_bias, uint8_t* wit_packed, uint8_t* in_range);

/* ---- Content-mode hash inputs from packed keys and raw messages (d = 256, q < 2^16 for lcb_content_str_batch).
 * In content mode (the Python layer's one_time_keys.set_content_str(True)) str() / repr() of a verification key or a
 * public statement is
 *     '<' + name + ' ' + SHAKE256(name || le16(secpar) || its int16 coefficient rows, little-endian).hexdigest(16) + '>'
 * with name OneTimeVerificationKey (rows: left, then right) or OneTimePublicStatement (one row): always 57 bytes.  Every
 * challenge message (lm_one_time_sigs.py:148, adaptor_sigs.py:176) and every BKLM aggregation message
 * (bklm_one_time_agg_sigs.py:65) contains such strings, so these three calls build the chmsg / agmsg inputs of every sign,
 * verify, adaptor and BKLM entry point above from packed keys without a host round trip. */
#define LCB_CONTENT_VK 0   /* packed uint8[n][2][32*bits]: left half, then right half */
#define LCB_CONTENT_ST 1   /* packed uint8[n][32*bits]                               */
/* Row i of out uint8[n][57] is exactly repr() of the key (kind LCB_CONTENT_VK) or statement (LCB_CONTENT_ST) whose NTT
 * form is lcb_unpack_batch(packed, bits, bias 0): unpack -> lcb_ntt_inv_batch -> the digest above over the centred int16
 * coefficients -> '<name ' + 32 lowercase hex digits + '>', for any input bytes (slots v >= q included); secpar is the
 * context's.  bits = 16 is the byte layout of a plain uint16 NTT array.  bits 1..16, packed buffer 4-byte aligned, at most
 * 2^30 items, n == 0 returns LCB_OK; LCB_ERR_INVALID with "the packed wire format is defined for d == 256, q < 2^16
 * contexts only" on any other context. */
int lcb_content_str_batch(lcb_ctx* ctx, int kind, const uint8_t* packed, int bits, int64_t n, uint8_t* out);
/* Challenge messages: item i of out is [st_str_i + ', '] + vk_str_i + ', ' + msg_i (st_str nullable: without it the LM
 * challenge str(otvk) + ', ' + msg, with it the adaptor challenge str(st) + ', ' + str(otvk) + ', ' + msg), at
 * out[out_off[i] .. out_off[i+1]), out_off[0] = 0.  st_str / vk_str uint8[n][57] (lcb_content_str_batch rows), msg ragged
 * (item i = msg[msg_off[i] .. msg_off[i+1]); msg_off[0] need not be 0).  The caller sizes out as
 * msg_off[n] - msg_off[0] + 59 n bytes, or + 118 n with st_str; out_off int64[n+1].  Pure byte assembly: valid on every
 * context.  At most 2^30 items. */
int lcb_challenge_inputs_batch(lcb_ctx* ctx, const uint8_t* st_str, const uint8_t* vk_str, const uint8_t* msg,
                               const int64_t* msg_off, int64_t n, uint8_t* out, int64_t* out_off);
/* BKLM aggregation messages: group g (its sorted items agg_off[g] .. agg_off[g+1], agg_off as in
 * lcb_bklm_aggregate_batch) is '[' + ', '.join("(" + vk_str + ", '" + msg + "')") + ']' over its items - str(list(zip(keys,
 * msgs))) for bitstring messages, '[]' for an empty group - at agmsg[agmsg_off[g] .. agmsg_off[g+1]), agmsg_off[0] = 0.
 * vk_str_sorted uint8[total][57], msg_sorted ragged as in lcb_challenge_inputs_batch (msg_off int64[total+1]); message
 * bytes are written as given.  Group g takes 2 + sum(63 + len_i) + 2 max(count_g - 1, 0) bytes; agmsg_off int64[n_agg+1].
 * At most 2^30 items.  The challenge messages of the same items come from lcb_challenge_inputs_batch on the same arrays. */
int lcb_aggregation_inputs_batch(lcb_ctx* ctx, const int64_t* agg_off, int64_t n_agg, const uint8_t* vk_str_sorted,
                                 const uint8_t* msg_sorted, const int64_t* msg_off, uint8_t* agmsg, int64_t* agmsg_off);

/* ---- Multi-device context: ONE call shards a HOST-resident batch over several GPUs of the box (SURVEY.md 8(b), 8(e)).
 * devices[] lists CUDA ordinals (an ordinal may repeat: two contexts on one GPU).  Independent units (keygen, sign,
 * verify) are split into contiguous ranges by the reference's distribute_tasks rule (lm_one_time_sigs.py:194-215: the
 * first n % ndev shards are one longer), one host thread per device, no data-path communication.  BKLM aggregate /
 * aggregate_verify (bklm_one_time_agg_sigs.py:92-116) shard the SORTED list; the per-device int32 partial sums are
 * gathered on device 0 by peer copies (NVLink where peer access exists), added by a kernel and finished there - the
 * exchange step that lattice_cryptography_b200/distributed.py performs with one NCCL reduce when there is one
 * process per GPU.  Every data pointer of these calls must be HOST memory; device-resident work goes through the
 * per-device contexts (lcb_mctx_ctx).  Arguments are those of the single-device calls. */
typedef struct lcb_mctx lcb_mctx;
int lcb_mctx_create(lcb_mctx** out, const int* devices, int ndev, int secpar, int q, int d, int l);
int lcb_mctx_destroy(lcb_mctx* m);
int lcb_mctx_ndev(const lcb_mctx* m);
lcb_ctx* lcb_mctx_ctx(lcb_mctx* m, int i);
const char* lcb_mctx_last_error(const lcb_mctx* m);
int lcb_mctx_set_key_ch(lcb_mctx* m, const int16_t* key_ch_coef);
int lcb_mctx_lm_keygen_batch(lcb_mctx* m, const lcb_scheme* sch, const uint8_t* seeds, const int64_t* seed_off, int64_t n,
                             int16_t* sk_coef, uint16_t* sk_ntt, uint16_t* vk_ntt, int16_t* vk_coef);
int lcb_mctx_lm_sign_batch(lcb_mctx* m, const lcb_scheme* sch, const uint16_t* sk_ntt, const uint8_t* chmsg,
                           const int64_t* chmsg_off, int64_t n, int16_t* sig);
int lcb_mctx_lm_verify_batch(lcb_mctx* m, const lcb_scheme* sch, const uint16_t* vk_ntt, const uint8_t* chmsg,
                             const int64_t* chmsg_off, const int16_t* sig, const uint16_t* st_ntt, int64_t n, int bd,
                             int wt, uint8_t* verdict);
int lcb_mctx_lm_verify_packed_batch(lcb_mctx* m, const lcb_scheme* sch, const uint8_t* vk_packed, int vk_bits,
                                    const uint8_t* chmsg, const int64_t* chmsg_off, const uint8_t* sig_packed,
                                    int sig_bits, int sig_bias, int64_t n, int bd, int wt, uint8_t* verdict);
/* whole aggregate / aggregate_verify in one call: coefficient derivation, sharded sums, device-side reduce, finish */
int lcb_mctx_bklm_aggregate(lcb_mctx* m, const lcb_scheme* sch, const int16_t* sig_sorted, const uint8_t* agmsg,
                            int64_t agmsg_len, int64_t n, int16_t* ag_sig);
int lcb_mctx_bklm_aggregate_verify(lcb_mctx* m, const lcb_scheme* sch, const uint16_t* vk_ntt_sorted,
                                   const uint8_t* chmsg_sorted, const int64_t* chmsg_off, const uint8_t* agmsg,
                                   int64_t agmsg_len, int64_t n, const int16_t* ag_sig, int ag_cap, int avf_bd,
                                   int avf_wt, uint8_t* verdict);

/* Instrumentation: kernels launched by this ctx since creation (bench.py's gpu_launches). */
int64_t lcb_launch_count(const lcb_ctx* ctx);
/* Optional per-kernel timing with CUDA events on the ctx stream (what bench.py's roofline reads).
 * kernel names: sampler shake256 ntt_fwd ntt_inv poly_mul matvec sign verify vec_addsub agg_coefs
 * agg_partial agg_finish aggv_partial aggv_finish pack unpack, and for the batch calls group_ids agg_coefs_seg
 * agg_partial_seg aggv_partial_seg aggv_residues aggv_limits, and agg_finish_pack for packed aggregates.  The fused packed
 * routes are counted under the kernel they extend: packed signing (from NTT-form or packed signing keys) under sign, packed
 * verification (including witness verification on packed witnesses) under verify, adapt / extract on packed witnesses
 * under vec_addsub.  The content-mode hash inputs: content_str (after unpack and ntt_inv), challenge_inputs, and
 * group_ids + aggregation_inputs.
 * lcb_profile_read synchronises the stream. */
int lcb_profile_enable(lcb_ctx* ctx, int on);
int lcb_profile_reset(lcb_ctx* ctx);
int lcb_profile_read(lcb_ctx* ctx, const char* kernel, double* total_ms, int64_t* launches);

#ifdef __cplusplus
}
#endif
#endif /* LCB200_H */
