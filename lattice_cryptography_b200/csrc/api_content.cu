// api_content.cu — content-mode hash inputs of the C ABI (content.cu): the content strings of packed keys and
// statements, and the challenge and aggregation hash inputs built from them and the raw messages; the per-group sort of
// content strings and the row / ragged gathers that put a batch into that order (order.cu).
#include <cstdlib>

#include "api_internal.h"

using namespace lcb;
using namespace lcb::abi;

namespace {

// off[0] and off[n] of a ragged offset array on the host.  A host array is checked (never decreases, starts at >= 0); a
// device array is trusted, as every device offset array of this ABI, and costs one 16-byte read.
int offset_ends(lcb_ctx* c, const int64_t* off, int64_t n, int64_t* first, int64_t* last, const char* what) {
    if (on_device(off)) {
        CK(c, cudaMemcpyAsync(first, off, sizeof(int64_t), cudaMemcpyDeviceToHost, c->stream));
        CK(c, cudaMemcpyAsync(last, off + n, sizeof(int64_t), cudaMemcpyDeviceToHost, c->stream));
        CK(c, cudaStreamSynchronize(c->stream));
    } else {
        if (off[0] < 0) return fail(c, LCB_ERR_INVALID, std::string(what) + " must not be negative");
        for (int64_t i = 0; i < n; ++i)
            if (off[i + 1] < off[i]) return fail(c, LCB_ERR_INVALID, std::string(what) + " must not decrease");
        *first = off[0];
        *last = off[n];
    }
    if (*last < *first) return fail(c, LCB_ERR_INVALID, std::string(what) + " must not decrease");
    return LCB_OK;
}

// The message bytes msg[first .. last) on the device: a device blob is used in place (shift 0, the kernels index it with
// the caller's offsets); a host blob is staged from byte `first` on (shift = first).
int stage_messages(lcb_ctx* c, Staging& sg, const uint8_t* msg, int64_t first, int64_t last, const uint8_t** d_msg,
                   int64_t* shift) {
    *d_msg = msg;
    *shift = 0;
    if (last == first) return LCB_OK;
    if (!msg) return fail(c, LCB_ERR_INVALID, "message blob is NULL");
    if (on_device(msg)) return LCB_OK;
    *d_msg = sg.in(msg + first, (size_t)(last - first));
    *shift = first;
    return LCB_OK;
}

// a single int64 into a caller buffer, host or device
int put_offset(lcb_ctx* c, int64_t* dst, int64_t v) {
    CK(c, cudaMemcpyAsync(dst, &v, sizeof(int64_t), cudaMemcpyDefault, c->stream));
    CK(c, cudaStreamSynchronize(c->stream));
    return LCB_OK;
}

// Test knobs LCB_ORDER_SMALL_MAX / LCB_ORDER_BLOCK_MAX: the largest group of the per-item path (default 32) and of the
// per-block path (default ORDER_BLOCK_MAX) of lcb_content_order_batch, so that tests reach every path with small groups.
// They can only lower the defaults; negative values are ignored.
int order_limit(const char* name, int dflt) {
    if (const char* env = getenv(name)) {
        const long v = atol(env);
        if (v >= 0 && v < dflt) return (int)v;
    }
    return dflt;
}

// host index arrays are checked; device ones are trusted (the kernels treat an index outside [0, n_src) as empty)
int check_index(lcb_ctx* c, const int64_t* index, int64_t n, int64_t n_src) {
    if (on_device(index)) return LCB_OK;
    for (int64_t k = 0; k < n; ++k)
        if (index[k] < 0 || index[k] >= n_src) return fail(c, LCB_ERR_INVALID, "index outside [0, n_src)");
    return LCB_OK;
}

}  // namespace

extern "C" {

int lcb_content_str_batch(lcb_ctx* c, int kind, const uint8_t* packed, int bits, int64_t n, uint8_t* out) {
    LCB_RANGE();
    if (!c || !packed || !out || n < 0 || (kind != LCB_CONTENT_VK && kind != LCB_CONTENT_ST) || bits < 1 || bits > 16)
        return LCB_ERR_INVALID;
    if (int st = need_wire(c)) return st;
    if (int st = within_limit(c, n, "items in one content-string call")) return st;
    if (n == 0) return LCB_OK;
    CK(c, cudaSetDevice(c->device));
    const int rows = kind == LCB_CONTENT_VK ? 2 : 1;
    const char* name = kind == LCB_CONTENT_VK ? "OneTimeVerificationKey" : "OneTimePublicStatement";   // 22 bytes each
    uint8_t prefix[24], head[24];
    std::memcpy(prefix, name, 22);
    prefix[22] = (uint8_t)(c->secpar & 0xFF);
    prefix[23] = (uint8_t)((c->secpar >> 8) & 0xFF);
    head[0] = '<';
    std::memcpy(head + 1, name, 22);
    head[23] = ' ';
    const size_t row_bytes = (size_t)32 * bits;
    Staging sg(c);
    const uint8_t* d_in = sg.in(packed, (size_t)n * rows * row_bytes);
    uint8_t* d_out = sg.out(out, (size_t)n * 57);
    CK(c, sg.status());
    if (int st = need_aligned4(c, {d_in})) return st;
    // unpack -> inverse transform into engine scratch, in chunks of the packed keygen's size (four sampler waves)
    const int64_t wave = (int64_t)c->ring.num_sms * 5 * 128;
    const int64_t chunk = n < 4 * wave ? n : 4 * wave;
    uint16_t* d_ntt = sg.alloc<uint16_t>((size_t)chunk * rows * D);
    int16_t* d_coef = sg.alloc<int16_t>((size_t)chunk * rows * D);
    CK(c, sg.status());
    int st = for_chunks(n, chunk, [&](int64_t start, int64_t cnt, int64_t) -> int {
        CK(c, timed(c, K_UNPACK, [&] {
            return launch_unpack(c->ring, d_in + (size_t)start * rows * row_bytes, cnt * rows, bits, 0, d_ntt, c->stream);
        }));
        CK(c, timed(c, K_NTT_INV, [&] { return launch_ntt_inv(c->ring, d_ntt, cnt * rows, d_coef, c->stream); }));
        CK(c, timed(c, K_CONTENT_STR, [&] {
            return launch_content_str(c->ring, d_coef, cnt, rows, prefix, head, d_out + (size_t)start * 57, c->stream);
        }));
        return LCB_OK;
    });
    if (st != LCB_OK) return st;
    CK(c, sg.finish());
    return LCB_OK;
}

int lcb_challenge_inputs_batch(lcb_ctx* c, const uint8_t* st_str, const uint8_t* vk_str, const uint8_t* msg,
                               const int64_t* msg_off, int64_t n, uint8_t* out, int64_t* out_off) {
    LCB_RANGE();
    if (!c || !vk_str || !msg_off || !out || !out_off || n < 0) return LCB_ERR_INVALID;
    if (int st = within_limit(c, n, "items in one challenge-input call")) return st;
    CK(c, cudaSetDevice(c->device));
    if (n == 0) return put_offset(c, out_off, 0);
    int64_t first = 0, last = 0, shift = 0;
    int st = offset_ends(c, msg_off, n, &first, &last, "msg_off");
    if (st != LCB_OK) return st;
    const int64_t per = st_str ? 118 : 59;
    const int64_t out_len = (last - first) + n * per;
    Staging sg(c);
    const uint8_t* d_msg;
    st = stage_messages(c, sg, msg, first, last, &d_msg, &shift);
    if (st != LCB_OK) return st;
    const uint8_t* d_vk = sg.in(vk_str, (size_t)n * 57);
    const uint8_t* d_st = st_str ? sg.in(st_str, (size_t)n * 57) : nullptr;
    const int64_t* d_off = sg.in(msg_off, (size_t)n + 1);
    uint8_t* d_out = sg.out(out, (size_t)out_len);
    int64_t* d_out_off = sg.out(out_off, (size_t)n + 1);
    CK(c, sg.status());
    CK(c, timed(c, K_CHALLENGE_INPUTS, [&] {
        return launch_challenge_inputs(c->ring, d_st, d_vk, d_msg, shift, d_off, n, out_len, d_out, d_out_off, c->stream);
    }));
    CK(c, sg.finish());
    return LCB_OK;
}

int lcb_aggregation_inputs_batch(lcb_ctx* c, const int64_t* agg_off, int64_t n_agg, const uint8_t* vk_str_sorted,
                                 const uint8_t* msg_sorted, const int64_t* msg_off, uint8_t* agmsg, int64_t* agmsg_off) {
    LCB_RANGE();
    if (!c || !agg_off || !msg_off || !agmsg || !agmsg_off || n_agg < 0) return LCB_ERR_INVALID;
    if (int st = within_limit(c, n_agg, "aggregates in one call")) return st;
    CK(c, cudaSetDevice(c->device));
    if (n_agg == 0) return put_offset(c, agmsg_off, 0);
    // the group layout needs every group's item range and message bytes: both offset arrays on the host
    std::vector<int64_t> h_agg, h_moff;
    int64_t total = 0, mlast = 0;
    int st = read_offsets(c, agg_off, n_agg, false, true, &total, h_agg, "agg_off");
    if (st != LCB_OK) return st;
    if (total < 0 || total > ((int64_t)1 << 30)) return fail(c, LCB_ERR_INVALID, "at most 2^30 items per batch call");
    if (total > 0 && !vk_str_sorted) return LCB_ERR_INVALID;
    if (on_device(msg_off)) {
        h_moff.resize((size_t)total + 1);
        CK(c, cudaMemcpyAsync(h_moff.data(), msg_off, h_moff.size() * sizeof(int64_t), cudaMemcpyDeviceToHost, c->stream));
        CK(c, cudaStreamSynchronize(c->stream));
    } else {
        h_moff.assign(msg_off, msg_off + total + 1);
    }
    if (h_moff[0] < 0) return fail(c, LCB_ERR_INVALID, "msg_off must not be negative");
    for (int64_t i = 0; i < total; ++i)
        if (h_moff[(size_t)i + 1] < h_moff[(size_t)i]) return fail(c, LCB_ERR_INVALID, "msg_off must not decrease");
    mlast = h_moff[(size_t)total];
    // group g: 2 + sum(63 + len_i) + 2 * max(count_g - 1, 0) bytes
    std::vector<int64_t> h_ag((size_t)n_agg + 1, 0);
    for (int64_t g = 0; g < n_agg; ++g) {
        const int64_t a0 = h_agg[(size_t)g], a1 = h_agg[(size_t)g + 1], cnt = a1 - a0;
        if (a0 < 0 || cnt < 0 || a1 > total) return fail(c, LCB_ERR_INVALID, "agg_off must not decrease");
        h_ag[(size_t)g + 1] = h_ag[(size_t)g] + 2 + 63 * cnt + (h_moff[(size_t)a1] - h_moff[(size_t)a0]) + 2 * (cnt > 0 ? cnt - 1 : 0);
    }
    const int64_t out_len = h_ag[(size_t)n_agg];
    Staging sg(c);
    const uint8_t* d_msg;
    int64_t shift = 0;
    st = stage_messages(c, sg, msg_sorted, h_moff[0], mlast, &d_msg, &shift);
    if (st != LCB_OK) return st;
    const uint8_t* d_vk = sg.in(vk_str_sorted, (size_t)total * 57);
    const int64_t* d_agg = sg.in(agg_off, (size_t)n_agg + 1);
    const int64_t* d_moff = sg.in(msg_off, (size_t)total + 1);
    int64_t* d_ag = sg.alloc<int64_t>(h_ag.size());
    int32_t* d_gid = sg.alloc<int32_t>((size_t)total);
    uint8_t* d_out = sg.out(agmsg, (size_t)out_len);
    int64_t* d_ag_out = sg.out(agmsg_off, h_ag.size());
    CK(c, sg.status());
    CK(c, cudaMemcpyAsync(d_ag, h_ag.data(), h_ag.size() * sizeof(int64_t), cudaMemcpyHostToDevice, c->stream));
    CK(c, cudaMemcpyAsync(d_ag_out, d_ag, h_ag.size() * sizeof(int64_t), cudaMemcpyDeviceToDevice, c->stream));
    CK(c, timed(c, K_GROUP_IDS, [&] { return launch_group_ids(d_agg, n_agg, total, d_gid, c->ring.num_sms, c->stream); }));
    CK(c, timed(c, K_AGGREGATION_INPUTS, [&] {
        return launch_aggregation_inputs(c->ring, d_agg, d_ag, n_agg, d_gid, total, d_vk, d_msg, shift, d_moff, out_len, d_out,
                                         c->stream);
    }));
    CK(c, sg.finish());
    return LCB_OK;
}

int lcb_content_order_batch(lcb_ctx* c, const int64_t* agg_off, int64_t n_agg, const uint8_t* rows, int64_t* order) {
    LCB_RANGE();
    if (!c || !agg_off || n_agg < 0) return LCB_ERR_INVALID;
    if (int st = within_limit(c, n_agg, "aggregates in one call")) return st;
    if (n_agg == 0) return LCB_OK;
    CK(c, cudaSetDevice(c->device));
    // the group sizes choose the paths: the offsets are read on the host, and checked there whichever side they come from
    std::vector<int64_t> h_agg;
    int64_t total = 0;
    int st = read_offsets(c, agg_off, n_agg, false, true, &total, h_agg, "agg_off");
    if (st != LCB_OK) return st;
    if (h_agg[0] != 0) return fail(c, LCB_ERR_INVALID, "agg_off must start at 0");
    for (int64_t g = 0; g < n_agg; ++g)
        if (h_agg[(size_t)g + 1] < h_agg[(size_t)g]) return fail(c, LCB_ERR_INVALID, "agg_off must not decrease");
    if (total > ((int64_t)1 << 30)) return fail(c, LCB_ERR_INVALID, "at most 2^30 items per batch call");
    if (total == 0) return LCB_OK;
    if (!rows || !order) return LCB_ERR_INVALID;
    const int small_max = order_limit("LCB_ORDER_SMALL_MAX", 32);
    const int block_max = order_limit("LCB_ORDER_BLOCK_MAX", ORDER_BLOCK_MAX);
    bool any_small = false;
    std::vector<int32_t> blk;                                    // groups of the per-block path
    std::vector<int64_t> la0, lbase{0};                          // the largest groups: first item, concatenated position
    for (int64_t g = 0; g < n_agg; ++g) {
        const int64_t cnt = h_agg[(size_t)g + 1] - h_agg[(size_t)g];
        if (cnt == 0) continue;
        if (cnt <= small_max) {
            any_small = true;
        } else if (cnt <= block_max) {
            blk.push_back((int32_t)g);
        } else {
            la0.push_back(h_agg[(size_t)g]);
            lbase.push_back(lbase.back() + cnt);
        }
    }
    Staging sg(c);
    const uint8_t* d_rows = sg.in(rows, (size_t)total * 57);
    const int64_t* d_agg = sg.in(agg_off, (size_t)n_agg + 1);
    int64_t* d_order = sg.out(order, (size_t)total);
    CK(c, sg.status());
    if (any_small) {
        int32_t* d_gid = sg.alloc<int32_t>((size_t)total);
        CK(c, sg.status());
        CK(c, timed(c, K_GROUP_IDS, [&] { return launch_group_ids(d_agg, n_agg, total, d_gid, c->ring.num_sms, c->stream); }));
        CK(c, timed(c, K_CONTENT_ORDER, [&] {
            return launch_content_order_small(d_agg, d_gid, n_agg, total, d_rows, small_max, d_order, c->ring.num_sms, c->stream);
        }));
    }
    if (!blk.empty()) {
        const int32_t* d_blk = sg.in(blk.data(), blk.size());
        CK(c, sg.status());
        CK(c, timed(c, K_CONTENT_ORDER, [&] {
            return launch_content_order_block(d_agg, d_blk, (int64_t)blk.size(), n_agg, total, d_rows, d_order, c->stream);
        }));
    }
    if (!la0.empty()) {
        const int L = (int)la0.size();
        const int64_t m = lbase.back();
        size_t temp_bytes = 0;
        CK(c, content_order_large_scratch(m, &temp_bytes));
        const int64_t* d_a0 = sg.in(la0.data(), la0.size());
        const int64_t* d_base = sg.in(lbase.data(), lbase.size());
        uint64_t* d_keys = sg.alloc<uint64_t>((size_t)(2 * m));
        int32_t* d_perm = sg.alloc<int32_t>((size_t)(2 * m));
        uint8_t* d_temp = sg.alloc<uint8_t>(temp_bytes);
        CK(c, sg.status());
        CK(c, timed(c, K_CONTENT_ORDER, [&] {
            return launch_content_order_large(d_rows, total, d_a0, d_base, L, m, d_keys, d_perm, d_temp, temp_bytes, d_order,
                                              c->ring.num_sms, c->stream);
        }));
    }
    CK(c, sg.finish());
    return LCB_OK;
}

int lcb_gather_rows_batch(lcb_ctx* c, const uint8_t* src, int64_t n_src, int64_t row_bytes, const int64_t* index, int64_t n,
                          uint8_t* dst) {
    LCB_RANGE();
    if (!c || n < 0 || n_src < 0 || row_bytes < 1) return LCB_ERR_INVALID;
    if (int st = within_limit(c, n, "items in one gather call")) return st;
    if (n == 0) return LCB_OK;
    if (!index || !dst || (n_src > 0 && !src)) return LCB_ERR_INVALID;
    if (n_src > INT64_MAX / row_bytes || n > INT64_MAX / row_bytes) return fail(c, LCB_ERR_INVALID, "rows too large");
    CK(c, cudaSetDevice(c->device));
    if (int st = check_index(c, index, n, n_src)) return st;
    Staging sg(c);
    const uint8_t* d_src = sg.in(src, (size_t)(n_src * row_bytes));
    const int64_t* d_idx = sg.in(index, (size_t)n);
    uint8_t* d_dst = sg.out(dst, (size_t)(n * row_bytes));
    CK(c, sg.status());
    CK(c, timed(c, K_GATHER_ROWS, [&] {
        return launch_gather_rows(d_src, n_src, row_bytes, d_idx, n, d_dst, c->ring.num_sms, c->stream);
    }));
    CK(c, sg.finish());
    return LCB_OK;
}

int lcb_gather_ragged_batch(lcb_ctx* c, const uint8_t* blob, const int64_t* off, int64_t n_src, const int64_t* index, int64_t n,
                            uint8_t* out, int64_t out_cap, int64_t* out_off) {
    LCB_RANGE();
    if (!c || !off || !out_off || n < 0 || n_src < 0 || out_cap < 0) return LCB_ERR_INVALID;
    if (int st = within_limit(c, n, "items in one gather call")) return st;
    CK(c, cudaSetDevice(c->device));
    if (n == 0) return put_offset(c, out_off, 0);
    if (!index) return LCB_ERR_INVALID;
    if (int st = check_index(c, index, n, n_src)) return st;
    Staging sg(c);
    // a device blob with device offsets is used in place; otherwise the blob's extent off[0] .. off[n_src] is read (and
    // host offsets are checked) to stage it
    const uint8_t* d_blob = blob;
    int64_t shift = 0;
    if (!(on_device(off) && blob && on_device(blob))) {
        int64_t first = 0, last = 0;
        int st = offset_ends(c, off, n_src, &first, &last, "off");
        if (st != LCB_OK) return st;
        if ((st = stage_messages(c, sg, blob, first, last, &d_blob, &shift)) != LCB_OK) return st;
    }
    const int64_t* d_off = sg.in(off, (size_t)n_src + 1);
    const int64_t* d_idx = sg.in(index, (size_t)n);
    const int64_t tiles = ragged_scan_tiles(n);
    int64_t* d_tile = sg.alloc<int64_t>((size_t)tiles + 1);
    int64_t* d_out_off = sg.out(out_off, (size_t)n + 1);
    CK(c, sg.status());
    CK(c, timed(c, K_GATHER_RAGGED, [&] {
        return launch_ragged_scan(d_off, n_src, d_idx, n, d_tile, d_out_off, c->ring.num_sms, c->stream);
    }));
    // the one synchronisation of this call: the gathered total against out_cap, before anything is written to out
    int64_t need = 0;
    CK(c, cudaMemcpyAsync(&need, d_tile + tiles, sizeof(int64_t), cudaMemcpyDeviceToHost, c->stream));
    CK(c, cudaStreamSynchronize(c->stream));
    if (need > out_cap) return fail(c, LCB_ERR_INVALID, "the gathered items need more than out_cap bytes");
    if (need > 0 && !out) return LCB_ERR_INVALID;
    uint8_t* d_out = sg.out(out, (size_t)need);
    CK(c, sg.status());
    CK(c, timed(c, K_GATHER_RAGGED, [&] {
        return launch_gather_ragged(d_blob, shift, d_off, n_src, d_idx, n, d_out_off, need, d_out, c->ring.num_sms, c->stream);
    }));
    CK(c, sg.finish());
    return LCB_OK;
}

}  // extern "C"
