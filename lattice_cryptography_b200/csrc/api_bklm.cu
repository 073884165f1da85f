// api_bklm.cu — BKLM aggregation entry points of the C ABI: aggregation coefficients, the single-aggregate partial /
// finish steps, and batches of aggregates and aggregate verifications, on int16 arrays and on the packed wire format.
#include "api_internal.h"

using namespace lcb;
using namespace lcb::abi;

namespace {

int run_agg_coefs(lcb_ctx* c, const lcb_scheme* sch, const uint8_t* d_agmsg, int64_t agmsg_len, int64_t first,
                  int64_t count, int16_t* d_pairs) {
    SamplerArgs a{};
    int st = fill_sampler(c, a, salt_of(sch->ag_salt).c_str(), nullptr, sch->ag_bd, sch->ag_wt, 1);
    if (st != LCB_OK) return fail(c, st, "bad aggregation parameters");
    if (a.salt_len + 20 > 32) return fail(c, LCB_ERR_INVALID, "ag_salt longer than 12 bytes");
    a.msgs = d_agmsg;
    a.off = nullptr;
    a.n = count;
    a.shared_msg = 1;
    a.shared_len = agmsg_len;
    a.index_first = first;
    a.out_pairs = d_pairs;
    if (c->generic || sch->ag_wt != 1 || sch->ag_bd != 1) {
        // General aggregation coefficients (ag_wt > 1 or ag_bd > 1: bklm_one_time_agg_sigs.py:15-19 leaves both as
        // editable tables) and generic degrees: the full sampler over the shared message, one salt
        // ag_salt || str(index) per stream.
        uint8_t* salts = nullptr;
        int32_t* lens = nullptr;
        CK(c, cudaMallocAsync((void**)&salts, (size_t)count * SALT_BYTES, c->stream));
        cudaError_t e = cudaMallocAsync((void**)&lens, (size_t)count * sizeof(int32_t), c->stream);
        if (e != cudaSuccess) {
            cudaFreeAsync(salts, c->stream);
            return fail_cuda(c, e, "general aggregation coefficients");
        }
        e = launch_index_salts(a, salts, lens, c->stream);
        a.stream_salts = salts;
        a.stream_salt_len = lens;
        if (e == cudaSuccess) e = sampler_scratch(c, a);
        if (e == cudaSuccess) e = timed(c, K_AGG_COEFS, [&] { return launch_sampler(a, c->stream); });
        cudaFreeAsync(salts, c->stream);
        cudaFreeAsync(lens, c->stream);
        c->launches += 1;
        if (e != cudaSuccess) return fail_cuda(c, e, "general aggregation coefficients");
        return LCB_OK;
    }
    if (agg_coefs_two_lane(count, c->ring.num_sms)) {
        // few long streams: two lanes per sponge over the pre-split message (sampler.cu, k_agg_coefs_il)
        CK(c, grow(c, c->il_scratch, c->il_scratch_bytes, agg_il_bytes(agmsg_len)));
        a.il_msg = c->il_scratch;
        a.il_stride = agg_il_stride(agmsg_len);
        c->launches += 1;                                  // the pre-split kernel
    }
    CK(c, timed(c, K_AGG_COEFS, [&] { return launch_agg_coefs(a, c->ring.num_sms, c->stream); }));
    return LCB_OK;
}


// ---- batches of aggregates ------------------------------------------------------------------------------------
// What the host needs of the offset arrays of a batch call: the item and message totals, and for the per-group
// fallback every entry.  Host-resident arrays are checked (start at 0, never decrease; strictly increase when every
// group must hold a signature); device-resident ones are trusted, as every device offset array of this ABI, and only
// copied back as far as needed (one 8-byte read and a stream synchronisation for the totals).
struct GroupOffsets {
    int64_t items = 0, msg_bytes = 0;
    std::vector<int64_t> agg, msg;     // filled when `all`
    // the most items of one group (needs `all`)
    int64_t largest() const {
        int64_t most = 0;
        for (size_t g = 0; g + 1 < agg.size(); ++g) most = std::max(most, agg[g + 1] - agg[g]);
        return most;
    }
};

int group_offsets(lcb_ctx* c, const int64_t* agg_off, const int64_t* agmsg_off, int64_t n_agg, bool nonempty, bool all,
                  GroupOffsets& g) {
    int st = read_offsets(c, agg_off, n_agg, nonempty, all, &g.items, g.agg, "agg_off");
    if (st == LCB_OK) st = read_offsets(c, agmsg_off, n_agg, false, all, &g.msg_bytes, g.msg, "agmsg_off");
    if (st != LCB_OK) return st;
    if (g.items < 0 || g.items > ((int64_t)1 << 30)) return fail(c, LCB_ERR_INVALID, "at most 2^30 signatures per batch call");
    return LCB_OK;
}

// monomial aggregation coefficients (ag_wt = ag_bd = 1) on a d = 256 context: the segmented kernels of the fast route
bool fast_route(const lcb_ctx* c, const lcb_scheme* sch) { return !c->generic && sch->ag_wt == 1 && sch->ag_bd == 1; }

// The checks and offsets lcb_bklm_aggregate_batch and its packed twin share; n_agg == 0 returns LCB_OK with nothing read.
int aggregate_prologue(lcb_ctx* c, const lcb_scheme* sch, const int64_t* agg_off, const int64_t* agmsg_off, int64_t n_agg,
                       GroupOffsets& go) {
    if (int st = agg_params_ok(c, sch)) return st;
    if (int st = within_limit(c, n_agg, "aggregates in one call")) return st;
    if (n_agg == 0) return LCB_OK;
    CK(c, cudaSetDevice(c->device));
    return group_offsets(c, agg_off, agmsg_off, n_agg, true, !fast_route(c, sch), go);
}

// The checks and offsets lcb_bklm_aggregate_verify_batch and its packed twin share, up to the byte count of the challenge
// messages (needed only to stage a host blob); n_agg == 0 returns LCB_OK with nothing read.
int aggregate_verify_prologue(lcb_ctx* c, const lcb_scheme* sch, const int64_t* agg_off, const int64_t* agmsg_off,
                              int64_t n_agg, const void* vk, const uint8_t* chmsg, const int64_t* chmsg_off, const char* name,
                              GroupOffsets& go, int64_t* ch_bytes) {
    if (int st = agg_params_ok(c, sch)) return st;
    if (int st = need_key_ch(c, name)) return st;
    if (int st = within_limit(c, n_agg, "aggregates in one call")) return st;
    *ch_bytes = 0;
    if (n_agg == 0) return LCB_OK;
    CK(c, cudaSetDevice(c->device));
    int st = group_offsets(c, agg_off, agmsg_off, n_agg, false, !fast_route(c, sch), go);
    if (st != LCB_OK) return st;
    if (go.items == 0) return LCB_OK;
    if (!vk || !chmsg) return LCB_ERR_INVALID;
    std::vector<int64_t> unused;
    if (!on_device(chmsg_off) && (st = read_offsets(c, chmsg_off, go.items, false, false, ch_bytes, unused, "chmsg_off")) != LCB_OK)
        return st;
    CK(c, last_offset(c, chmsg, chmsg_off, go.items, ch_bytes));
    return LCB_OK;
}

// The aggregation-coefficient sampler arguments of the segmented kernel (ag_wt = ag_bd = 1)
int seg_coef_args(lcb_ctx* c, const lcb_scheme* sch, const uint8_t* d_msg, int64_t items, int16_t* d_pairs, SamplerArgs& a) {
    int st = fill_sampler(c, a, salt_of(sch->ag_salt).c_str(), nullptr, sch->ag_bd, sch->ag_wt, 1);
    if (st != LCB_OK) return fail(c, st, "bad aggregation parameters");
    if (a.salt_len + 20 > 32) return fail(c, LCB_ERR_INVALID, "ag_salt longer than 12 bytes");
    a.msgs = d_msg;
    a.n = items;
    a.out_pairs = d_pairs;
    return LCB_OK;
}

// The body of lcb_bklm_aggregate_batch over device buffers (go from group_offsets with all = !fast).  On the fast route
// (d = 256, monomial coefficients) the signatures may also be packed rows (sig_bits 11 / 13, bias sig_bias) and the
// aggregates may be written packed (ag_bits 1..16, bias ag_bias, in_range nullable); 0 bits = int16 arrays.
int aggregate_batch_dev(lcb_ctx* c, const lcb_scheme* sch, Staging& sg, const GroupOffsets& go, int64_t n_agg,
                        const void* d_sig, int sig_bits, int sig_bias, const uint8_t* d_msg, const int64_t* d_aoff,
                        const int64_t* d_moff, void* d_out, int ag_bits, int ag_bias, uint8_t* d_range) {
    const bool fast = fast_route(c, sch);
    if (!fast && (sig_bits || ag_bits)) return fail(c, LCB_ERR_INVALID, "packed aggregation needs monomial coefficients");
    const int l = c->l;
    const size_t D_ = (size_t)c->d * ew(c);
    const size_t pair_len = (size_t)sch->ag_wt * 2 * ew(c);
    int32_t* d_part = sg.alloc<int32_t>((size_t)n_agg * l * D_);
    // the fast route samples the coefficients of every item at once, the per-group route those of one group at a time
    int32_t* d_gid = fast ? sg.alloc<int32_t>((size_t)go.items) : nullptr;
    int16_t* d_pairs = sg.alloc<int16_t>((size_t)(fast ? go.items : go.largest()) * pair_len);
    CK(c, sg.status());
    CK(c, cudaMemsetAsync(d_part, 0, (size_t)n_agg * l * D_ * sizeof(int32_t), c->stream));
    if (fast) {
        SamplerArgs a{};
        int st = seg_coef_args(c, sch, d_msg, go.items, d_pairs, a);
        if (st != LCB_OK) return st;
        CK(c, timed(c, K_GROUP_IDS, [&] { return launch_group_ids(d_aoff, n_agg, go.items, d_gid, c->ring.num_sms, c->stream); }));
        CK(c, timed(c, K_AGG_COEFS_SEG, [&] { return launch_agg_coefs_seg(a, d_gid, d_aoff, d_moff, n_agg, c->stream); }));
        CK(c, timed(c, K_AGG_PARTIAL_SEG, [&] {
            return launch_agg_partial_seg(c->ring, d_sig, sig_bits, sig_bias, d_pairs, d_gid, go.items, n_agg, d_part, c->stream);
        }));
        if (ag_bits) {
            CK(c, timed(c, K_AGG_FINISH_PACK, [&] {
                return launch_agg_finish_pack(c->ring, d_part, n_agg * l, ag_bits, ag_bias, static_cast<uint8_t*>(d_out), d_range,
                                              c->stream);
            }));
        } else {
            CK(c, timed(c, K_AGG_FINISH, [&] {
                return launch_agg_finish_n(c->ring, d_part, n_agg * l * D, static_cast<int16_t*>(d_out), c->stream);
            }));
        }
        return LCB_OK;
    }
    // generic geometry or non-monomial coefficients: the single-aggregate kernels, group by group (correct, not fast)
    const bool monomial = sch->ag_wt == 1 && sch->ag_bd == 1;
    const int16_t* sig = static_cast<const int16_t*>(d_sig);
    int16_t* out = static_cast<int16_t*>(d_out);
    for (int64_t g = 0; g < n_agg; ++g) {
        const int64_t first = go.agg[(size_t)g], count = go.agg[(size_t)g + 1] - first;
        const int16_t* sig_g = sig + (size_t)first * l * D_;
        int32_t* part_g = d_part + (size_t)g * l * D_;
        if (count > 0) {
            int st = run_agg_coefs(c, sch, d_msg + go.msg[(size_t)g], go.msg[(size_t)g + 1] - go.msg[(size_t)g], 0, count, d_pairs);
            if (st != LCB_OK) return st;
            CK(c, timed(c, K_AGG_PARTIAL, [&] {
                if (!monomial) return g_launch_agg_partial_poly(c->gen, sig_g, d_pairs, sch->ag_wt, count, part_g, c->stream);
                return g_launch_agg_partial(c->gen, sig_g, d_pairs, count, part_g, c->stream);
            }));
        }
        CK(c, timed(c, K_AGG_FINISH, [&] {
            return c->generic ? g_launch_agg_finish(c->gen, part_g, out + (size_t)g * l * D_, c->stream)
                              : launch_agg_finish(c->ring, part_g, out + (size_t)g * l * D_, c->stream);
        }));
    }
    return LCB_OK;
}

// The body of lcb_bklm_aggregate_verify_batch over device buffers.  On the fast route the keys may also be 14-bit packed
// rows (vk_bits 14; 0 = uint16 slots, which the 16-bit packing is byte for byte) and the aggregates 12- / 14-bit packed
// rows with bias ag_bias (ag_bits 0 = int16).
int aggregate_verify_batch_dev(lcb_ctx* c, const lcb_scheme* sch, Staging& sg, const GroupOffsets& go, int64_t n_agg,
                               const void* d_vk, int vk_bits, const uint8_t* d_chmsg, const int64_t* d_choff,
                               const uint8_t* d_msg, const int64_t* d_aoff, const int64_t* d_moff, const void* d_ag, int ag_bits,
                               int ag_bias, int ag_cap, int avf_bd, int avf_wt, uint8_t* d_verdict) {
    const bool fast = fast_route(c, sch);
    if (!fast && (vk_bits || ag_bits)) return fail(c, LCB_ERR_INVALID, "packed aggregate verification needs monomial coefficients");
    const int l = c->l;
    const size_t D_ = (size_t)c->d * ew(c);
    const size_t pair_len = (size_t)sch->ag_wt * 2 * ew(c);
    int16_t* d_ch = sg.alloc<int16_t>((size_t)go.items * sch->ch_wt * 2 * ew(c));
    int32_t* d_part = sg.alloc<int32_t>((size_t)n_agg * D_);
    int32_t* d_gid = fast ? sg.alloc<int32_t>((size_t)go.items) : nullptr;
    int16_t* d_pairs = sg.alloc<int16_t>((size_t)(fast ? go.items : go.largest()) * pair_len);
    uint16_t* d_rhs = fast ? sg.alloc<uint16_t>((size_t)n_agg * D) : nullptr;
    CK(c, sg.status());
    CK(c, cudaMemsetAsync(d_part, 0, (size_t)n_agg * D_ * sizeof(int32_t), c->stream));
    int st;
    if (go.items > 0) {           // the challenges of every item of every group: one sampler launch
        st = run_challenge(c, sch, d_chmsg, d_choff, go.items, d_ch);
        if (st != LCB_OK) return st;
    }
    if (fast) {
        SamplerArgs a{};
        st = seg_coef_args(c, sch, d_msg, go.items, d_pairs, a);
        if (st != LCB_OK) return st;
        CK(c, timed(c, K_GROUP_IDS, [&] { return launch_group_ids(d_aoff, n_agg, go.items, d_gid, c->ring.num_sms, c->stream); }));
        CK(c, timed(c, K_AGG_COEFS_SEG, [&] { return launch_agg_coefs_seg(a, d_gid, d_aoff, d_moff, n_agg, c->stream); }));
        CK(c, timed(c, K_AGGV_PARTIAL_SEG, [&] {
            return launch_aggv_partial_seg(c->ring, d_vk, vk_bits, d_ch, sch->ch_wt, d_pairs, d_gid, go.items, n_agg, d_part,
                                           c->stream);
        }));
        CK(c, timed(c, K_AGGV_RESIDUES, [&] { return launch_aggv_residues(c->ring, d_part, n_agg * D, d_rhs, c->stream); }));
        // bounds and key_ch * ag_sig == rhs: the witness-verify form of k_verify.  Every int16 passes a bound of 32768, as
        // it passes any larger one in k_aggv_finish.
        CK(c, timed(c, K_VERIFY, [&] {
            if (ag_bits)
                return launch_verify_rhs_packed(c->ring, static_cast<const uint8_t*>(d_ag), ag_bits, ag_bias, d_rhs, n_agg,
                                                std::min(avf_bd, 32768), avf_wt, d_verdict, c->stream);
            return launch_verify(c->ring, static_cast<const int16_t*>(d_ag), nullptr, nullptr, 0, d_rhs, nullptr, n_agg,
                                 std::min(avf_bd, 32768), avf_wt, d_verdict, c->stream);
        }));
        CK(c, timed(c, K_AGGV_LIMITS, [&] {
            if (ag_bits)
                return launch_aggv_limits_packed(c->ring, d_aoff, n_agg, static_cast<const uint8_t*>(d_ag), ag_bits, ag_bias, ag_cap,
                                                 d_verdict, c->stream);
            return launch_aggv_limits(c->ring, d_aoff, n_agg, static_cast<const int16_t*>(d_ag), ag_cap, d_verdict, c->stream);
        }));
        return LCB_OK;
    }
    // generic geometry or non-monomial coefficients: the single-aggregate kernels, group by group (correct, not fast)
    const bool monomial = sch->ag_wt == 1 && sch->ag_bd == 1;
    const uint16_t* vk = static_cast<const uint16_t*>(d_vk);
    const int16_t* ag = static_cast<const int16_t*>(d_ag);
    for (int64_t g = 0; g < n_agg; ++g) {
        const int64_t first = go.agg[(size_t)g], count = go.agg[(size_t)g + 1] - first;
        int32_t* part_g = d_part + (size_t)g * D_;
        const int16_t* ag_g = ag + (size_t)g * l * D_;
        if (count > 0) {
            const uint16_t* vk_g = vk + (size_t)first * 2 * D_;
            const int16_t* ch_g = d_ch + (size_t)first * sch->ch_wt * 2 * ew(c);
            st = run_agg_coefs(c, sch, d_msg + go.msg[(size_t)g], go.msg[(size_t)g + 1] - go.msg[(size_t)g], 0, count, d_pairs);
            if (st != LCB_OK) return st;
            CK(c, timed(c, K_AGGV_PARTIAL, [&] {
                if (!monomial)
                    return g_launch_aggv_partial_poly(c->gen, vk_g, ch_g, sch->ch_wt, d_pairs, sch->ag_wt, count, part_g, c->stream);
                return g_launch_aggv_partial(c->gen, vk_g, ch_g, sch->ch_wt, d_pairs, count, part_g, c->stream);
            }));
        }
        CK(c, timed(c, K_AGGV_FINISH, [&] {
            return c->generic ? g_launch_aggv_finish(c->gen, part_g, ag_g, count, ag_cap, avf_bd, avf_wt, d_verdict + g, c->stream)
                              : launch_aggv_finish(c->ring, part_g, ag_g, count, ag_cap, avf_bd, avf_wt, d_verdict + g, c->stream);
        }));
    }
    return LCB_OK;
}

}  // namespace

extern "C" {

int lcb_bklm_agg_coefs(lcb_ctx* c, const lcb_scheme* sch, const uint8_t* agmsg, int64_t agmsg_len, int64_t first,
                       int64_t count, int16_t* out_pairs) {
    LCB_RANGE();
    if (!c || !sch || !agmsg || !out_pairs || agmsg_len < 0 || first < 0 || count < 0) return LCB_ERR_INVALID;
    if (count == 0) return LCB_OK;
    CK(c, cudaSetDevice(c->device));
    Staging sg(c);
    const uint8_t* d_msg = sg.in(agmsg, (size_t)agmsg_len);
    int16_t* d_pairs = sg.out(out_pairs, (size_t)count * sch->ag_wt * 2 * ew(c));
    CK(c, sg.status());
    int st = run_agg_coefs(c, sch, d_msg, agmsg_len, first, count, d_pairs);
    if (st != LCB_OK) return st;
    CK(c, sg.finish());
    return LCB_OK;
}

int lcb_bklm_aggregate_partial(lcb_ctx* c, const lcb_scheme* sch, const int16_t* sig_sorted, const int16_t* ag_pairs,
                               const uint8_t* agmsg, int64_t agmsg_len, int64_t first, int64_t count,
                               int32_t* partial) {
    LCB_RANGE();
    if (!c || !sch || !partial || count < 0 || (count > 0 && !sig_sorted) || (!ag_pairs && !agmsg)) return LCB_ERR_INVALID;
    CK(c, cudaSetDevice(c->device));
    const int l = c->l;
    const size_t D_ = (size_t)c->d * ew(c);
    const size_t pair_len = (size_t)sch->ag_wt * 2 * ew(c);
    const bool monomial = sch->ag_wt == 1 && sch->ag_bd == 1;
    if (int st = agg_params_ok(c, sch)) return st;
    Staging sg(c);
    const int16_t* d_sig = sg.in(sig_sorted, (size_t)count * l * D_);
    const int16_t* d_pairs = sg.in(ag_pairs, (size_t)count * pair_len);
    int32_t* d_partial = sg.out(partial, (size_t)l * c->d * ew(c));
    CK(c, sg.status());
    CK(c, cudaMemsetAsync(d_partial, 0, (size_t)l * c->d * ew(c) * sizeof(int32_t), c->stream));
    if (count > 0) {
        if (!d_pairs) {
            const uint8_t* d_msg = sg.in(agmsg, (size_t)agmsg_len);
            int16_t* d_coefs = sg.alloc<int16_t>((size_t)count * pair_len);
            CK(c, sg.status());
            int st = run_agg_coefs(c, sch, d_msg, agmsg_len, first, count, d_coefs);
            if (st != LCB_OK) return st;
            d_pairs = d_coefs;
        }
        CK(c, timed(c, K_AGG_PARTIAL, [&] {
            if (!monomial) return g_launch_agg_partial_poly(c->gen, d_sig, d_pairs, sch->ag_wt, count, d_partial, c->stream);
            return c->generic ? g_launch_agg_partial(c->gen, d_sig, d_pairs, count, d_partial, c->stream)
                              : launch_agg_partial(c->ring, d_sig, d_pairs, count, d_partial, c->stream);
        }));
    }
    CK(c, sg.finish());
    return LCB_OK;
}

int lcb_bklm_aggregate_finish(lcb_ctx* c, const int32_t* partial_sum, int16_t* ag_sig) {
    LCB_RANGE();
    if (!c || !partial_sum || !ag_sig) return LCB_ERR_INVALID;
    CK(c, cudaSetDevice(c->device));
    Staging sg(c);
    const int32_t* d_partial = sg.in(partial_sum, (size_t)c->l * c->d * ew(c));
    int16_t* d_out = sg.out(ag_sig, (size_t)c->l * c->d * ew(c));
    CK(c, sg.status());
    CK(c, timed(c, K_AGG_FINISH, [&] {
        return c->generic ? g_launch_agg_finish(c->gen, d_partial, d_out, c->stream) : launch_agg_finish(c->ring, d_partial, d_out, c->stream);
    }));
    CK(c, sg.finish());
    return LCB_OK;
}

int lcb_bklm_aggverify_partial(lcb_ctx* c, const lcb_scheme* sch, const uint16_t* vk_ntt_sorted,
                               const uint8_t* chmsg_sorted, const int64_t* chmsg_off, const int16_t* ag_pairs,
                               const uint8_t* agmsg, int64_t agmsg_len, int64_t first, int64_t count,
                               int32_t* partial) {
    LCB_RANGE();
    if (!c || !sch || !partial || count < 0 || (count > 0 && (!vk_ntt_sorted || !chmsg_off)) || (!ag_pairs && !agmsg))
        return LCB_ERR_INVALID;
    CK(c, cudaSetDevice(c->device));
    const size_t D_ = (size_t)c->d * ew(c);
    const size_t pair_len = (size_t)sch->ag_wt * 2 * ew(c);
    const bool monomial = sch->ag_wt == 1 && sch->ag_bd == 1;
    if (int st = agg_params_ok(c, sch)) return st;
    Staging sg(c);
    int32_t* d_partial = sg.out(partial, (size_t)c->d * ew(c));
    CK(c, sg.status());
    CK(c, cudaMemsetAsync(d_partial, 0, (size_t)c->d * ew(c) * sizeof(int32_t), c->stream));
    if (count > 0) {
        int64_t total = 0;
        CK(c, last_offset(c, chmsg_sorted, chmsg_off, count, &total));
        const uint16_t* d_vk = sg.in(vk_ntt_sorted, (size_t)count * 2 * D_);
        const uint8_t* d_chmsg = sg.in(chmsg_sorted, (size_t)total);
        const int64_t* d_off = sg.in(chmsg_off, (size_t)count + 1);
        const int16_t* d_ag = sg.in(ag_pairs, (size_t)count * pair_len);
        int16_t* d_ch = sg.alloc<int16_t>((size_t)count * sch->ch_wt * 2 * ew(c));
        CK(c, sg.status());
        int st = run_challenge(c, sch, d_chmsg, d_off, count, d_ch);
        if (st != LCB_OK) return st;
        if (!d_ag) {
            const uint8_t* d_agmsg = sg.in(agmsg, (size_t)agmsg_len);
            int16_t* d_pairs = sg.alloc<int16_t>((size_t)count * pair_len);
            CK(c, sg.status());
            st = run_agg_coefs(c, sch, d_agmsg, agmsg_len, first, count, d_pairs);
            if (st != LCB_OK) return st;
            d_ag = d_pairs;
        }
        CK(c, timed(c, K_AGGV_PARTIAL, [&] {
            if (!monomial) return g_launch_aggv_partial_poly(c->gen, d_vk, d_ch, sch->ch_wt, d_ag, sch->ag_wt, count, d_partial, c->stream);
            return c->generic ? g_launch_aggv_partial(c->gen, d_vk, d_ch, sch->ch_wt, d_ag, count, d_partial, c->stream)
                              : launch_aggv_partial(c->ring, d_vk, d_ch, sch->ch_wt, d_ag, count, d_partial, c->stream);
        }));
    }
    CK(c, sg.finish());
    return LCB_OK;
}

int lcb_bklm_aggverify_finish(lcb_ctx* c, const int32_t* partial_sum, const int16_t* ag_sig, int64_t total, int ag_cap,
                              int avf_bd, int avf_wt, uint8_t* verdict) {
    LCB_RANGE();
    if (!c || !partial_sum || !ag_sig || !verdict) return LCB_ERR_INVALID;
    if (int st = need_key_ch(c, "lcb_bklm_aggverify_finish")) return st;
    CK(c, cudaSetDevice(c->device));
    Staging sg(c);
    const int32_t* d_partial = sg.in(partial_sum, (size_t)c->d * ew(c));
    const int16_t* d_sig = sg.in(ag_sig, (size_t)c->l * c->d * ew(c));
    uint8_t* d_verdict = sg.out(verdict, 1);
    CK(c, sg.status());
    CK(c, timed(c, K_AGGV_FINISH, [&] {
        return c->generic ? g_launch_aggv_finish(c->gen, d_partial, d_sig, total, ag_cap, avf_bd, avf_wt, d_verdict, c->stream)
                          : launch_aggv_finish(c->ring, d_partial, d_sig, total, ag_cap, avf_bd, avf_wt, d_verdict, c->stream);
    }));
    CK(c, sg.finish());
    return LCB_OK;
}

int lcb_bklm_aggregate_batch(lcb_ctx* c, const lcb_scheme* sch, const int64_t* agg_off, int64_t n_agg,
                             const int16_t* sig_sorted, const uint8_t* agmsg, const int64_t* agmsg_off, int16_t* ag_sig) {
    LCB_RANGE();
    if (!c || !sch || !agg_off || !agmsg_off || n_agg < 0 || (n_agg > 0 && (!sig_sorted || !agmsg || !ag_sig)))
        return LCB_ERR_INVALID;
    GroupOffsets go;
    int st = aggregate_prologue(c, sch, agg_off, agmsg_off, n_agg, go);
    if (st != LCB_OK || n_agg == 0) return st;
    const int l = c->l;
    const size_t D_ = (size_t)c->d * ew(c);
    Staging sg(c);
    const int16_t* d_sig = sg.in(sig_sorted, (size_t)go.items * l * D_);
    const uint8_t* d_msg = sg.in(agmsg, (size_t)go.msg_bytes);
    const int64_t* d_aoff = sg.in(agg_off, (size_t)n_agg + 1);
    const int64_t* d_moff = sg.in(agmsg_off, (size_t)n_agg + 1);
    int16_t* d_out = sg.out(ag_sig, (size_t)n_agg * l * D_);
    CK(c, sg.status());
    st = aggregate_batch_dev(c, sch, sg, go, n_agg, d_sig, 0, 0, d_msg, d_aoff, d_moff, d_out, 0, 0, nullptr);
    if (st != LCB_OK) return st;
    CK(c, sg.finish());
    return LCB_OK;
}

int lcb_bklm_aggregate_verify_batch(lcb_ctx* c, const lcb_scheme* sch, const int64_t* agg_off, int64_t n_agg,
                                    const uint16_t* vk_ntt_sorted, const uint8_t* chmsg_sorted, const int64_t* chmsg_off,
                                    const uint8_t* agmsg, const int64_t* agmsg_off, const int16_t* ag_sig, int ag_cap,
                                    int avf_bd, int avf_wt, uint8_t* verdict) {
    LCB_RANGE();
    if (!c || !sch || !agg_off || !agmsg_off || !chmsg_off || n_agg < 0 || (n_agg > 0 && (!agmsg || !ag_sig || !verdict)))
        return LCB_ERR_INVALID;
    GroupOffsets go;
    int64_t ch_bytes;
    int st = aggregate_verify_prologue(c, sch, agg_off, agmsg_off, n_agg, vk_ntt_sorted, chmsg_sorted, chmsg_off,
                                       "lcb_bklm_aggregate_verify_batch", go, &ch_bytes);
    if (st != LCB_OK || n_agg == 0) return st;
    const int l = c->l;
    const size_t D_ = (size_t)c->d * ew(c);
    Staging sg(c);
    const uint16_t* d_vk = sg.in(vk_ntt_sorted, (size_t)go.items * 2 * D_);
    const uint8_t* d_chmsg = sg.in(chmsg_sorted, (size_t)ch_bytes);
    const int64_t* d_choff = sg.in(chmsg_off, (size_t)go.items + 1);
    const uint8_t* d_msg = sg.in(agmsg, (size_t)go.msg_bytes);
    const int64_t* d_aoff = sg.in(agg_off, (size_t)n_agg + 1);
    const int64_t* d_moff = sg.in(agmsg_off, (size_t)n_agg + 1);
    const int16_t* d_ag = sg.in(ag_sig, (size_t)n_agg * l * D_);
    uint8_t* d_verdict = sg.out(verdict, (size_t)n_agg);
    CK(c, sg.status());
    st = aggregate_verify_batch_dev(c, sch, sg, go, n_agg, d_vk, 0, d_chmsg, d_choff, d_msg, d_aoff, d_moff, d_ag, 0, 0, ag_cap,
                                    avf_bd, avf_wt, d_verdict);
    if (st != LCB_OK) return st;
    CK(c, sg.finish());
    return LCB_OK;
}

// lcb_bklm_aggregate_batch on packed signatures, writing packed aggregates.  Fused route (monomial coefficients, 11- or
// 13-bit signatures, 16-byte aligned signature rows): k_agg_partial_seg expands the packed rows itself and
// k_agg_finish_pack writes the packed aggregates.  Anything else is unpacked into scratch first, aggregated by the code
// of lcb_bklm_aggregate_batch and packed by k_pack.
int lcb_bklm_aggregate_packed_batch(lcb_ctx* c, const lcb_scheme* sch, const int64_t* agg_off, int64_t n_agg,
                                    const uint8_t* sig_packed, int sig_bits, int sig_bias, const uint8_t* agmsg,
                                    const int64_t* agmsg_off, int ag_bits, int ag_bias, uint8_t* ag_packed, uint8_t* in_range) {
    LCB_RANGE();
    if (!c || !sch || !agg_off || !agmsg_off || n_agg < 0 || (n_agg > 0 && (!sig_packed || !agmsg || !ag_packed)) ||
        !wire_args_ok(sig_bits, sig_bias) || !wire_args_ok(ag_bits, ag_bias))
        return LCB_ERR_INVALID;
    if (int st = need_wire(c)) return st;
    GroupOffsets go;
    int st = aggregate_prologue(c, sch, agg_off, agmsg_off, n_agg, go);
    if (st != LCB_OK || n_agg == 0) return st;
    const int l = c->l;
    Staging sg(c);
    const uint8_t* d_sigp = sg.in(sig_packed, (size_t)go.items * l * 32 * sig_bits);
    const uint8_t* d_msg = sg.in(agmsg, (size_t)go.msg_bytes);
    const int64_t* d_aoff = sg.in(agg_off, (size_t)n_agg + 1);
    const int64_t* d_moff = sg.in(agmsg_off, (size_t)n_agg + 1);
    uint8_t* d_agp = sg.out(ag_packed, (size_t)n_agg * l * 32 * ag_bits);
    uint8_t* d_range = sg.out(in_range, (size_t)n_agg * l);
    CK(c, sg.status());
    if ((st = need_aligned4(c, {d_sigp, d_agp}))) return st;
    // the fused route reads signature rows with 16-byte loads: a caller-owned device buffer that is only 4-byte aligned
    // takes the unpack-first route
    if (fast_route(c, sch) && (sig_bits == 11 || sig_bits == 13) && aligned16({d_sigp})) {
        st = aggregate_batch_dev(c, sch, sg, go, n_agg, d_sigp, sig_bits, sig_bias, d_msg, d_aoff, d_moff, d_agp, ag_bits,
                                 ag_bias, d_range);
    } else {
        int16_t* d_sig = sg.alloc<int16_t>((size_t)go.items * l * D);
        int16_t* d_ag = sg.alloc<int16_t>((size_t)n_agg * l * D);
        CK(c, sg.status());
        CK(c, timed(c, K_UNPACK, [&] { return launch_unpack(c->ring, d_sigp, go.items * l, sig_bits, sig_bias, d_sig, c->stream); }));
        st = aggregate_batch_dev(c, sch, sg, go, n_agg, d_sig, 0, 0, d_msg, d_aoff, d_moff, d_ag, 0, 0, nullptr);
        if (st == LCB_OK)
            CK(c, timed(c, K_PACK, [&] { return launch_pack(c->ring, d_ag, n_agg * l, ag_bits, ag_bias, d_agp, d_range, c->stream); }));
    }
    if (st != LCB_OK) return st;
    CK(c, sg.finish());
    return LCB_OK;
}

// lcb_bklm_aggregate_verify_batch on packed keys and aggregates.  Fused route (monomial coefficients, 14- or 16-bit keys,
// 12- or 14-bit aggregates, 16-byte aligned aggregate rows and 16-bit key rows): k_aggv_partial_seg reads the packed
// keys, k_verify (witness form) and k_aggv_limits_packed the packed aggregates.  Anything else is unpacked into scratch
// first and verified by the code of lcb_bklm_aggregate_verify_batch.
int lcb_bklm_aggregate_verify_packed_batch(lcb_ctx* c, const lcb_scheme* sch, const int64_t* agg_off, int64_t n_agg,
                                           const uint8_t* vk_packed, int vk_bits, const uint8_t* chmsg_sorted,
                                           const int64_t* chmsg_off, const uint8_t* agmsg, const int64_t* agmsg_off,
                                           const uint8_t* ag_packed, int ag_bits, int ag_bias, int ag_cap, int avf_bd,
                                           int avf_wt, uint8_t* verdict) {
    LCB_RANGE();
    if (!c || !sch || !agg_off || !agmsg_off || !chmsg_off || n_agg < 0 || (n_agg > 0 && (!agmsg || !ag_packed || !verdict)) ||
        !wire_args_ok(vk_bits, 0) || !wire_args_ok(ag_bits, ag_bias))
        return LCB_ERR_INVALID;
    if (int st = need_wire(c)) return st;
    GroupOffsets go;
    int64_t ch_bytes;
    int st = aggregate_verify_prologue(c, sch, agg_off, agmsg_off, n_agg, vk_packed, chmsg_sorted, chmsg_off,
                                       "lcb_bklm_aggregate_verify_packed_batch", go, &ch_bytes);
    if (st != LCB_OK || n_agg == 0) return st;
    const int l = c->l;
    Staging sg(c);
    const uint8_t* d_vkp = sg.in(vk_packed, (size_t)go.items * 2 * 32 * vk_bits);
    const uint8_t* d_chmsg = sg.in(chmsg_sorted, (size_t)ch_bytes);
    const int64_t* d_choff = sg.in(chmsg_off, (size_t)go.items + 1);
    const uint8_t* d_msg = sg.in(agmsg, (size_t)go.msg_bytes);
    const int64_t* d_aoff = sg.in(agg_off, (size_t)n_agg + 1);
    const int64_t* d_moff = sg.in(agmsg_off, (size_t)n_agg + 1);
    const uint8_t* d_agp = sg.in(ag_packed, (size_t)n_agg * l * 32 * ag_bits);
    uint8_t* d_verdict = sg.out(verdict, (size_t)n_agg);
    CK(c, sg.status());
    if ((st = need_aligned4(c, {d_vkp, d_agp}))) return st;
    // the fused route stages aggregate rows with 16-byte cp.async and reads 16-bit key rows with 128-bit loads: a
    // caller-owned device buffer that is only 4-byte aligned takes the unpack-first route
    if (fast_route(c, sch) && aligned16({d_agp, vk_bits == 14 ? nullptr : d_vkp}) && (vk_bits == 14 || vk_bits == 16) &&
        (ag_bits == 12 || ag_bits == 14)) {
        st = aggregate_verify_batch_dev(c, sch, sg, go, n_agg, d_vkp, vk_bits == 14 ? 14 : 0, d_chmsg, d_choff, d_msg, d_aoff,
                                        d_moff, d_agp, ag_bits, ag_bias, ag_cap, avf_bd, avf_wt, d_verdict);
    } else {
        uint16_t* d_vk = sg.alloc<uint16_t>((size_t)go.items * 2 * D);
        int16_t* d_ag = sg.alloc<int16_t>((size_t)n_agg * l * D);
        CK(c, sg.status());
        CK(c, timed(c, K_UNPACK, [&] { return launch_unpack(c->ring, d_vkp, go.items * 2, vk_bits, 0, d_vk, c->stream); }));
        CK(c, timed(c, K_UNPACK, [&] { return launch_unpack(c->ring, d_agp, n_agg * l, ag_bits, ag_bias, d_ag, c->stream); }));
        st = aggregate_verify_batch_dev(c, sch, sg, go, n_agg, d_vk, 0, d_chmsg, d_choff, d_msg, d_aoff, d_moff, d_ag, 0, 0, ag_cap,
                                        avf_bd, avf_wt, d_verdict);
    }
    if (st != LCB_OK) return st;
    CK(c, sg.finish());
    return LCB_OK;
}

}  // extern "C"
