// api_adaptor.cu — adaptor-signature entry points of the C ABI: witness generation (plain and packed), adapt / extract on
// the wire format (with int16 or packed witnesses) and witness verification (plain and packed).
#include "api_internal.h"

using namespace lcb;
using namespace lcb::abi;

namespace {

// The body of lcb_adaptor_witgen_batch (wp == null: one pass over the whole batch) and of lcb_adaptor_witgen_packed_batch
// (wp set, every unpacked output null: chunks of kWireChunkPoly / l witnesses in secret scratch).
int witgen(lcb_ctx* c, const lcb_scheme* sch, const uint8_t* seeds, const int64_t* seed_off, int64_t n, int16_t* wit_coef,
           uint16_t* st_ntt, int16_t* st_coef, const PackedOut* wp, const char* name) {
    if (int st = need_key_ch(c, name)) return st;
    if (n == 0) return LCB_OK;
    CK(c, cudaSetDevice(c->device));
    const int l = c->l;
    SamplerArgs a{};
    int st = fill_sampler(c, a, salt_of(sch->wit_salt).c_str(), nullptr, sch->wit_bd, sch->wit_wt, l);
    if (st != LCB_OK) return fail(c, st, "bad witness parameters");
    int64_t total = 0;
    CK(c, last_offset(c, seeds, seed_off, n, &total));
    const size_t D_ = (size_t)c->d * ew(c);
    Staging sg(c);
    const uint8_t* d_seeds = sg.in(seeds, (size_t)total);
    const int64_t* d_off = sg.in(seed_off, (size_t)n + 1);
    int16_t* d_wit = sg.out(wit_coef, (size_t)n * l * D_, true);
    uint16_t* d_st_ntt = sg.out(st_ntt, (size_t)n * D_);
    int16_t* d_st_coef = sg.out(st_coef, (size_t)n * D_);
    uint8_t* d_witp = wp ? sg.out(wp->rows, (size_t)n * l * 32 * wp->bits, true) : nullptr;
    uint8_t* d_witr = wp ? sg.out(wp->in_range, (size_t)n * l) : nullptr;
    uint8_t* d_stp = wp ? sg.out(wp->pub, (size_t)n * 32 * wp->pub_bits) : nullptr;
    CK(c, sg.status());
    if ((st = need_aligned4(c, {d_witp, d_stp}))) return st;
    const int64_t chunk = wp && n > kWireChunkPoly / l ? kWireChunkPoly / l : n;
    int16_t* scratch = d_wit ? nullptr : sg.alloc<int16_t>((size_t)chunk * l * D_, true);
    // NTT-form statements of a chunk, to be packed
    uint16_t* st_scratch = d_stp ? sg.alloc<uint16_t>((size_t)chunk * D_) : nullptr;
    CK(c, sg.status());
    st = for_chunks(n, chunk, [&](int64_t start, int64_t cnt, int64_t) -> int {
        int16_t* wit = d_wit ? d_wit + start * l * D_ : scratch;
        // the sampler writes only the wit_wt nonzero coefficients of each polynomial
        if (sch->wit_wt < c->d) CK(c, cudaMemsetAsync(wit, 0, (size_t)cnt * l * D_ * sizeof(int16_t), c->stream));
        a.msgs = d_seeds;
        a.off = d_off + start;
        a.n = cnt;
        a.out_dense = wit;
        a.dense_stride = (int64_t)l * c->d;
        CK(c, sampler_scratch(c, a));
        CK(c, timed(c, K_SAMPLER, [&] { return launch_sampler(a, c->stream); }));
        uint16_t* o_st = d_st_ntt ? d_st_ntt + start * D_ : st_scratch;
        int16_t* o_stc = d_st_coef ? d_st_coef + start * D_ : nullptr;
        CK(c, timed(c, K_MATVEC, [&] {
            return c->generic ? g_launch_matvec(c->gen, wit, cnt, nullptr, o_st, o_stc, c->stream)
                              : launch_matvec(c->ring, wit, cnt, nullptr, o_st, o_stc, c->stream);
        }));
        if (d_witp)
            CK(c, timed(c, K_PACK, [&] {
                return launch_pack(c->ring, wit, cnt * l, wp->bits, wp->bias, d_witp + start * l * 32 * wp->bits,
                                   d_witr ? d_witr + start * l : nullptr, c->stream);
            }));
        if (d_stp)
            CK(c, timed(c, K_PACK, [&] {
                return launch_pack(c->ring, st_scratch, cnt, wp->pub_bits, 0, d_stp + start * 32 * wp->pub_bits, nullptr, c->stream);
            }));
        return LCB_OK;
    });
    if (st != LCB_OK) return st;
    CK(c, sg.finish());
    return LCB_OK;
}

// adapt / extract with packed witnesses: unpack both -> k_vec_addsub -> pack in ONE kernel (k_addsub_packed, every width),
// counted under vec_addsub.  a = presig (adapt) or sig (extract), b = wit (adapt) or presig (extract).
int addsub_packed(lcb_ctx* c, const uint8_t* a, int a_bits, int a_bias, bool a_secret, const uint8_t* b, int b_bits, int b_bias,
                  bool b_secret, int sub, int64_t npoly, int bits, int bias, bool out_secret, uint8_t* out, uint8_t* in_range) {
    if (!c || !a || !b || !out || npoly < 0 || !wire_args_ok(a_bits, a_bias) || !wire_args_ok(b_bits, b_bias) ||
        !wire_args_ok(bits, bias))
        return LCB_ERR_INVALID;
    if (int st = need_wire(c)) return st;
    if (npoly == 0) return LCB_OK;
    CK(c, cudaSetDevice(c->device));
    Staging sg(c);
    const uint8_t* d_a = sg.in(a, (size_t)npoly * 32 * a_bits, a_secret);
    const uint8_t* d_b = sg.in(b, (size_t)npoly * 32 * b_bits, b_secret);
    uint8_t* d_out = sg.out(out, (size_t)npoly * 32 * bits, out_secret);
    uint8_t* d_range = sg.out(in_range, (size_t)npoly);
    CK(c, sg.status());
    if (int st = need_aligned4(c, {d_a, d_b, d_out})) return st;
    CK(c, timed(c, K_ADDSUB, [&] {
        return launch_addsub_packed(c->ring, d_a, a_bits, a_bias, d_b, b_bits, b_bias, sub, npoly, bits, bias, d_out, d_range,
                                    c->stream);
    }));
    CK(c, sg.finish());
    return LCB_OK;
}

}  // namespace

extern "C" {

int lcb_adaptor_witgen_batch(lcb_ctx* c, const lcb_scheme* sch, const uint8_t* seeds, const int64_t* seed_off,
                             int64_t n, int16_t* wit_coef, uint16_t* st_ntt, int16_t* st_coef) {
    LCB_RANGE();
    if (!c || !sch || !seed_off || n < 0) return LCB_ERR_INVALID;
    return witgen(c, sch, seeds, seed_off, n, wit_coef, st_ntt, st_coef, nullptr, "lcb_adaptor_witgen_batch");
}

// lcb_adaptor_witgen_batch -> lcb_pack_batch (witnesses, coefficient form) and lcb_pack_batch (statements, NTT form, bias 0),
// chunk by chunk inside the witgen loop: the 16-bit witnesses never leave engine scratch.
int lcb_adaptor_witgen_packed_batch(lcb_ctx* c, const lcb_scheme* sch, const uint8_t* seeds, const int64_t* seed_off,
                                    int64_t n, int wit_bits, int wit_bias, uint8_t* wit_packed, uint8_t* wit_in_range,
                                    int st_bits, uint8_t* st_packed) {
    LCB_RANGE();
    if (!c || !sch || !seed_off || n < 0 || (!wit_packed && !st_packed) || !wire_args_ok(wit_bits, wit_bias) ||
        !wire_args_ok(st_bits, 0))
        return LCB_ERR_INVALID;
    if (int st = need_wire(c)) return st;
    if (int st = within_limit(c, n, "items in one witgen call")) return st;
    const PackedOut wp{wit_bits, wit_bias, wit_packed, wit_packed ? wit_in_range : nullptr, st_bits, st_packed};
    return witgen(c, sch, seeds, seed_off, n, nullptr, nullptr, nullptr, &wp, "lcb_adaptor_witgen_packed_batch");
}

// adapt / extract on the wire format: unpack -> k_vec_addsub -> (pack), in chunks of bounded int16 scratch.  HBM streams of
// a few thousand operations per signature, so they are composed from the existing kernels and exact by construction.
int lcb_adaptor_adapt_packed_batch(lcb_ctx* c, const uint8_t* presig_packed, int presig_bits, int presig_bias,
                                   const int16_t* wit_coef, int64_t npoly, int sig_bits, int sig_bias, uint8_t* sig_packed,
                                   uint8_t* in_range) {
    LCB_RANGE();
    if (!c || !presig_packed || !wit_coef || !sig_packed || npoly < 0 || !wire_args_ok(presig_bits, presig_bias) ||
        !wire_args_ok(sig_bits, sig_bias))
        return LCB_ERR_INVALID;
    if (int st = need_wire(c)) return st;
    if (npoly == 0) return LCB_OK;
    CK(c, cudaSetDevice(c->device));
    Staging sg(c);
    const uint8_t* d_prep = sg.in(presig_packed, (size_t)npoly * 32 * presig_bits);
    const int16_t* d_wit = sg.in(wit_coef, (size_t)npoly * D, true);
    uint8_t* d_sigp = sg.out(sig_packed, (size_t)npoly * 32 * sig_bits);
    uint8_t* d_range = sg.out(in_range, (size_t)npoly);
    CK(c, sg.status());
    if (int st = need_aligned4(c, {d_prep, d_sigp})) return st;
    const int64_t chunk = npoly < kWireChunkPoly ? npoly : kWireChunkPoly;
    int16_t* d_pre = sg.alloc<int16_t>((size_t)chunk * D);
    int16_t* d_sig = sg.alloc<int16_t>((size_t)chunk * D);
    CK(c, sg.status());
    int st = for_chunks(npoly, chunk, [&](int64_t first, int64_t m, int64_t) -> int {
        CK(c, timed(c, K_UNPACK, [&] {
            return launch_unpack(c->ring, d_prep + (size_t)first * 32 * presig_bits, m, presig_bits, presig_bias, d_pre,
                                 c->stream);
        }));
        CK(c, timed(c, K_ADDSUB, [&] { return launch_vec_addsub(c->ring, d_pre, d_wit + (size_t)first * D, m * D, 0, d_sig, c->stream); }));
        CK(c, timed(c, K_PACK, [&] {
            return launch_pack(c->ring, d_sig, m, sig_bits, sig_bias, d_sigp + (size_t)first * 32 * sig_bits,
                               d_range ? d_range + first : nullptr, c->stream);
        }));
        return LCB_OK;
    });
    if (st != LCB_OK) return st;
    CK(c, sg.finish());
    return LCB_OK;
}

int lcb_adaptor_extract_packed_batch(lcb_ctx* c, const uint8_t* sig_packed, int sig_bits, int sig_bias,
                                     const uint8_t* presig_packed, int presig_bits, int presig_bias, int64_t npoly,
                                     int16_t* wit_coef) {
    LCB_RANGE();
    if (!c || !sig_packed || !presig_packed || !wit_coef || npoly < 0 || !wire_args_ok(sig_bits, sig_bias) ||
        !wire_args_ok(presig_bits, presig_bias))
        return LCB_ERR_INVALID;
    if (int st = need_wire(c)) return st;
    if (npoly == 0) return LCB_OK;
    CK(c, cudaSetDevice(c->device));
    Staging sg(c);
    const uint8_t* d_sigp = sg.in(sig_packed, (size_t)npoly * 32 * sig_bits);
    const uint8_t* d_prep = sg.in(presig_packed, (size_t)npoly * 32 * presig_bits);
    int16_t* d_wit = sg.out(wit_coef, (size_t)npoly * D, true);
    CK(c, sg.status());
    if (int st = need_aligned4(c, {d_sigp, d_prep})) return st;
    const int64_t chunk = npoly < kWireChunkPoly ? npoly : kWireChunkPoly;
    int16_t* d_sig = sg.alloc<int16_t>((size_t)chunk * D);
    int16_t* d_pre = sg.alloc<int16_t>((size_t)chunk * D);
    CK(c, sg.status());
    int st = for_chunks(npoly, chunk, [&](int64_t first, int64_t m, int64_t) -> int {
        CK(c, timed(c, K_UNPACK, [&] {
            return launch_unpack(c->ring, d_sigp + (size_t)first * 32 * sig_bits, m, sig_bits, sig_bias, d_sig, c->stream);
        }));
        CK(c, timed(c, K_UNPACK, [&] {
            return launch_unpack(c->ring, d_prep + (size_t)first * 32 * presig_bits, m, presig_bits, presig_bias, d_pre,
                                 c->stream);
        }));
        CK(c, timed(c, K_ADDSUB, [&] { return launch_vec_addsub(c->ring, d_sig, d_pre, m * D, 1, d_wit + (size_t)first * D, c->stream); }));
        return LCB_OK;
    });
    if (st != LCB_OK) return st;
    CK(c, sg.finish());
    return LCB_OK;
}

int lcb_adaptor_adapt_packed_wit_batch(lcb_ctx* c, const uint8_t* presig_packed, int presig_bits, int presig_bias,
                                       const uint8_t* wit_packed, int wit_bits, int wit_bias, int64_t npoly, int sig_bits,
                                       int sig_bias, uint8_t* sig_packed, uint8_t* in_range) {
    LCB_RANGE();
    return addsub_packed(c, presig_packed, presig_bits, presig_bias, false, wit_packed, wit_bits, wit_bias, true, 0, npoly,
                         sig_bits, sig_bias, false, sig_packed, in_range);
}

int lcb_adaptor_extract_packed_wit_batch(lcb_ctx* c, const uint8_t* sig_packed, int sig_bits, int sig_bias,
                                         const uint8_t* presig_packed, int presig_bits, int presig_bias, int64_t npoly,
                                         int wit_bits, int wit_bias, uint8_t* wit_packed, uint8_t* in_range) {
    LCB_RANGE();
    return addsub_packed(c, sig_packed, sig_bits, sig_bias, false, presig_packed, presig_bits, presig_bias, false, 1, npoly,
                         wit_bits, wit_bias, true, wit_packed, in_range);
}

int lcb_adaptor_witness_verify_batch(lcb_ctx* c, const int16_t* wit_coef, const uint16_t* st_ntt, int64_t n, int bd,
                                     int wt, uint8_t* verdict) {
    LCB_RANGE();
    if (!c || !wit_coef || !st_ntt || !verdict || n < 0 || bd < 0 || wt < 0) return LCB_ERR_INVALID;
    if (int st = need_key_ch(c, "lcb_adaptor_witness_verify_batch")) return st;
    if (int st = within_limit(c, n, "items in one verify call")) return st;
    if (n == 0) return LCB_OK;
    CK(c, cudaSetDevice(c->device));
    Staging sg(c);
    const int16_t* d_wit = sg.in(wit_coef, (size_t)n * c->l * c->d * ew(c));
    const uint16_t* d_st = sg.in(st_ntt, (size_t)n * c->d * ew(c));
    uint8_t* d_verdict = sg.out(verdict, (size_t)n);
    CK(c, sg.status());
    CK(c, timed(c, K_VERIFY, [&] {
        return c->generic ? g_launch_verify(c->gen, d_wit, nullptr, nullptr, 0, d_st, nullptr, n, bd, wt, d_verdict, c->stream)
                          : launch_verify(c->ring, d_wit, nullptr, nullptr, 0, d_st, nullptr, n, bd > 32767 ? 32767 : bd, wt, d_verdict,
                                          c->stream);
    }));
    CK(c, sg.finish());
    return LCB_OK;
}

// unpack witnesses and statements -> lcb_adaptor_witness_verify_batch.  Fused route (witness / statement widths 2 / 14,
// 12 / 14, 2 / 16, 14 / 16 with statements at the key width ceil(log2 q); 16-byte aligned witness rows and 16-bit
// statement rows): k_verify reads both packed rows directly.  Anything else unpacks chunks of kWireChunkPoly / l items into
// secret scratch and runs the witness-verify launch on them.
int lcb_adaptor_witness_verify_packed_batch(lcb_ctx* c, const uint8_t* wit_packed, int wit_bits, int wit_bias,
                                            const uint8_t* st_packed, int st_bits, int64_t n, int bd, int wt,
                                            uint8_t* verdict) {
    LCB_RANGE();
    if (!c || !wit_packed || !st_packed || !verdict || n < 0 || bd < 0 || wt < 0 || !wire_args_ok(wit_bits, wit_bias) ||
        !wire_args_ok(st_bits, 0))
        return LCB_ERR_INVALID;
    if (int st = need_wire(c)) return st;
    if (int st = need_key_ch(c, "lcb_adaptor_witness_verify_packed_batch")) return st;
    if (int st = within_limit(c, n, "items in one verify call")) return st;
    if (n == 0) return LCB_OK;
    CK(c, cudaSetDevice(c->device));
    const int l = c->l;
    const size_t wit_item = (size_t)l * 32 * wit_bits;
    Staging sg(c);
    const uint8_t* d_witp = sg.in(wit_packed, (size_t)n * wit_item, true);
    const uint8_t* d_stp = sg.in(st_packed, (size_t)n * 32 * st_bits);
    uint8_t* d_verdict = sg.out(verdict, (size_t)n);
    CK(c, sg.status());
    if (int st = need_aligned4(c, {d_witp, d_stp})) return st;
    const int bd_k = bd > 32767 ? 32767 : bd;
    // k_verify stages witness rows with 16-byte cp.async and reads 16-bit statement rows with 128-bit loads: a caller-owned
    // device buffer that is only 4-byte aligned takes the composed route
    const bool fused = aligned16({d_witp, st_bits == 14 ? nullptr : d_stp}) && st_bits == ceil_log2(c->q) &&
                       ((st_bits == 14 && (wit_bits == 2 || wit_bits == 12)) || (st_bits == 16 && (wit_bits == 2 || wit_bits == 14)));
    if (fused) {
        CK(c, timed(c, K_VERIFY, [&] {
            return launch_verify_rhs_packed(c->ring, d_witp, wit_bits, wit_bias, reinterpret_cast<const uint16_t*>(d_stp), n,
                                            bd_k, wt, d_verdict, c->stream, st_bits);
        }));
    } else {
        const int64_t chunk = n < kWireChunkPoly / l ? n : kWireChunkPoly / l;
        int16_t* d_wit = sg.alloc<int16_t>((size_t)chunk * l * D, true);
        uint16_t* d_st = sg.alloc<uint16_t>((size_t)chunk * D);
        CK(c, sg.status());
        int st = for_chunks(n, chunk, [&](int64_t first, int64_t m, int64_t) -> int {
            CK(c, timed(c, K_UNPACK, [&] {
                return launch_unpack(c->ring, d_witp + (size_t)first * wit_item, m * l, wit_bits, wit_bias, d_wit, c->stream);
            }));
            CK(c, timed(c, K_UNPACK, [&] {
                return launch_unpack(c->ring, d_stp + (size_t)first * 32 * st_bits, m, st_bits, 0, d_st, c->stream);
            }));
            CK(c, timed(c, K_VERIFY, [&] {
                return launch_verify(c->ring, d_wit, nullptr, nullptr, 0, d_st, nullptr, m, bd_k, wt, d_verdict + first,
                                     c->stream);
            }));
            return LCB_OK;
        });
        if (st != LCB_OK) return st;
    }
    CK(c, sg.finish());
    return LCB_OK;
}

}  // extern "C"
