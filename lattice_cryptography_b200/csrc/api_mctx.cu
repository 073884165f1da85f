// api_mctx.cu — the multi-device context of the C ABI (lcb_mctx_*).
#include <thread>

#include "api_internal.h"

using namespace lcb;
using namespace lcb::abi;

// ================================================================================================================
// Multi-device context (SURVEY.md 8(b): `devices[], ndev`; 8(e)): ONE call shards a host-resident batch over all
// GPUs of the box.  Independent units (keygen / sign / verify) are split into contiguous ranges - the reference's
// distribute_tasks rule, lm_one_time_sigs.py:194-215: the first n % ndev shards are one longer - and run on one
// host thread per device with no data-path communication.  BKLM aggregate / aggregate_verify shard the SORTED
// list, every device reduces its shard to an int32 partial sum in its own memory, the partial sums travel to device
// 0 as peer copies (NVLink when peer access is available) and are added there by a kernel before the finish step.
// One process per GPU with torch.distributed / NCCL (lattice_cryptography_b200/distributed.py, bench.py) remains the
// way to scale across processes; this is the single-process route for C callers.
struct lcb_mctx {
    std::vector<lcb_ctx*> ctx;
    std::string last_error;
};

namespace {

__global__ void k_partial_add(int64_t n, int wide, void* __restrict__ acc, const void* __restrict__ add) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    if (wide) static_cast<long long*>(acc)[i] += static_cast<const long long*>(add)[i];
    else static_cast<int32_t*>(acc)[i] += static_cast<const int32_t*>(add)[i];
}

struct Shard { int64_t first, count; };

Shard shard_of(int64_t n, int i, int parts) {
    const int64_t base = n / parts, extra = n % parts;
    return {i * base + (i < extra ? i : extra), base + (i < extra ? 1 : 0)};
}

// fn(i, ctx_i, shard_i) on one host thread per device; first failure wins
template <typename F>
int on_all(lcb_mctx* m, int64_t n, F&& fn) {
    const int parts = (int)m->ctx.size();
    std::vector<int> status(parts, LCB_OK);
    std::vector<std::thread> th;
    for (int i = 0; i < parts; ++i)
        th.emplace_back([&, i] { status[i] = fn(i, m->ctx[i], shard_of(n, i, parts)); });
    for (auto& t : th) t.join();
    for (int i = 0; i < parts; ++i)
        if (status[i] != LCB_OK) {
            m->last_error = "device shard " + std::to_string(i) + ": " + m->ctx[i]->last_error;
            return status[i];
        }
    return LCB_OK;
}

// offsets of one shard rebased to its own blob start
std::vector<int64_t> rebased(const int64_t* off, const Shard& s) {
    std::vector<int64_t> o((size_t)s.count + 1);
    for (int64_t k = 0; k <= s.count; ++k) o[(size_t)k] = off[s.first + k] - off[s.first];
    return o;
}

template <typename T>
T* at(T* p, size_t elems) { return p ? p + elems : nullptr; }

// partial sums of all devices -> device 0 (peer copies) -> added by k_partial_add; returns the device-0 buffer
int reduce_partials(lcb_mctx* m, std::vector<void*>& part, size_t words) {
    lcb_ctx* c0 = m->ctx[0];
    const size_t bytes = words * sizeof(int32_t) * ew(c0);
    CK(c0, cudaSetDevice(c0->device));
    void* tmp = nullptr;
    CK(c0, cudaMalloc(&tmp, bytes));
    for (size_t i = 1; i < part.size(); ++i) {
        CK(c0, cudaMemcpyPeerAsync(tmp, c0->device, part[i], m->ctx[i]->device, bytes, c0->stream));
        k_partial_add<<<(unsigned)((words + 255) / 256), 256, 0, c0->stream>>>((int64_t)words, c0->wide ? 1 : 0, part[0], tmp);
        CK(c0, cudaGetLastError());
        c0->launches += 1;
    }
    CK(c0, cudaStreamSynchronize(c0->stream));
    cudaFree(tmp);
    return LCB_OK;
}

bool host_only(lcb_mctx* m, std::initializer_list<const void*> ptrs) {
    for (const void* p : ptrs)
        if (p && on_device(p)) {
            m->last_error = "lcb_mctx_* entry points shard HOST buffers; pass device buffers to the per-device contexts (lcb_mctx_ctx)";
            return false;
        }
    return true;
}

}  // namespace

extern "C" {

int lcb_mctx_create(lcb_mctx** out, const int* devices, int ndev, int secpar, int q, int d, int l) {
    if (!out || !devices || ndev < 1 || ndev > 64) return LCB_ERR_INVALID;
    *out = nullptr;
    lcb_mctx* m = new (std::nothrow) lcb_mctx();
    if (!m) return LCB_ERR_OOM;
    for (int i = 0; i < ndev; ++i) {
        lcb_ctx* c = nullptr;
        const int st = lcb_ctx_create(&c, devices[i], secpar, q, d, l);
        if (st != LCB_OK) {
            for (lcb_ctx* x : m->ctx) lcb_ctx_destroy(x);
            delete m;
            return st;
        }
        m->ctx.push_back(c);
    }
    for (int i = 1; i < ndev; ++i)          // best effort: peer copies fall back to staging through the host without it
        if (devices[i] != devices[0]) {
            int can = 0;
            if (cudaDeviceCanAccessPeer(&can, devices[0], devices[i]) == cudaSuccess && can) {
                cudaSetDevice(devices[0]);
                if (cudaDeviceEnablePeerAccess(devices[i], 0) != cudaSuccess) cudaGetLastError();
            }
        }
    *out = m;
    return LCB_OK;
}

int lcb_mctx_destroy(lcb_mctx* m) {
    if (!m) return LCB_OK;
    for (lcb_ctx* c : m->ctx) lcb_ctx_destroy(c);
    delete m;
    return LCB_OK;
}

int lcb_mctx_ndev(const lcb_mctx* m) { return m ? (int)m->ctx.size() : LCB_ERR_INVALID; }

lcb_ctx* lcb_mctx_ctx(lcb_mctx* m, int i) { return (m && i >= 0 && i < (int)m->ctx.size()) ? m->ctx[i] : nullptr; }

const char* lcb_mctx_last_error(const lcb_mctx* m) { return m ? m->last_error.c_str() : ""; }

int lcb_mctx_set_key_ch(lcb_mctx* m, const int16_t* key_ch_coef) {
    if (!m || !key_ch_coef) return LCB_ERR_INVALID;
    for (lcb_ctx* c : m->ctx) {
        const int st = lcb_set_key_ch(c, key_ch_coef);
        if (st != LCB_OK) { m->last_error = c->last_error; return st; }
    }
    return LCB_OK;
}

int lcb_mctx_lm_keygen_batch(lcb_mctx* m, const lcb_scheme* sch, const uint8_t* seeds, const int64_t* seed_off, int64_t n,
                             int16_t* sk_coef, uint16_t* sk_ntt, uint16_t* vk_ntt, int16_t* vk_coef) {
    LCB_RANGE();
    if (!m || !sch || !seeds || !seed_off || n < 0) return LCB_ERR_INVALID;
    if (!host_only(m, {seeds, seed_off, sk_coef, sk_ntt, vk_ntt, vk_coef})) return LCB_ERR_INVALID;
    return on_all(m, n, [&](int, lcb_ctx* c, Shard s) {
        const size_t D_ = (size_t)c->d * ew(c), f = (size_t)s.first;
        const std::vector<int64_t> off = rebased(seed_off, s);
        return lcb_lm_keygen_batch(c, sch, seeds + seed_off[s.first], off.data(), s.count, at(sk_coef, f * 2 * c->l * D_),
                                   at(sk_ntt, f * 2 * c->l * D_), at(vk_ntt, f * 2 * D_), at(vk_coef, f * 2 * D_));
    });
}

int lcb_mctx_lm_sign_batch(lcb_mctx* m, const lcb_scheme* sch, const uint16_t* sk_ntt, const uint8_t* chmsg,
                           const int64_t* chmsg_off, int64_t n, int16_t* sig) {
    LCB_RANGE();
    if (!m || !sch || !sk_ntt || !chmsg_off || !sig || n < 0) return LCB_ERR_INVALID;
    if (!host_only(m, {sk_ntt, chmsg, chmsg_off, sig})) return LCB_ERR_INVALID;
    return on_all(m, n, [&](int, lcb_ctx* c, Shard s) {
        const size_t D_ = (size_t)c->d * ew(c), f = (size_t)s.first;
        const std::vector<int64_t> off = rebased(chmsg_off, s);
        return lcb_lm_sign_batch(c, sch, sk_ntt + f * 2 * c->l * D_, chmsg + chmsg_off[s.first], off.data(), s.count,
                                 sig + f * c->l * D_);
    });
}

int lcb_mctx_lm_verify_batch(lcb_mctx* m, const lcb_scheme* sch, const uint16_t* vk_ntt, const uint8_t* chmsg,
                             const int64_t* chmsg_off, const int16_t* sig, const uint16_t* st_ntt, int64_t n, int bd, int wt,
                             uint8_t* verdict) {
    LCB_RANGE();
    if (!m || !sch || !vk_ntt || !chmsg_off || !sig || !verdict || n < 0) return LCB_ERR_INVALID;
    if (!host_only(m, {vk_ntt, chmsg, chmsg_off, sig, st_ntt, verdict})) return LCB_ERR_INVALID;
    return on_all(m, n, [&](int, lcb_ctx* c, Shard s) {
        const size_t D_ = (size_t)c->d * ew(c), f = (size_t)s.first;
        const std::vector<int64_t> off = rebased(chmsg_off, s);
        return lcb_lm_verify_batch(c, sch, vk_ntt + f * 2 * D_, chmsg + chmsg_off[s.first], off.data(), sig + f * c->l * D_,
                                   st_ntt ? st_ntt + f * D_ : nullptr, s.count, bd, wt, verdict + f);
    });
}

int lcb_mctx_lm_verify_packed_batch(lcb_mctx* m, const lcb_scheme* sch, const uint8_t* vk_packed, int vk_bits,
                                    const uint8_t* chmsg, const int64_t* chmsg_off, const uint8_t* sig_packed, int sig_bits,
                                    int sig_bias, int64_t n, int bd, int wt, uint8_t* verdict) {
    LCB_RANGE();
    if (!m || !sch || !vk_packed || !chmsg_off || !sig_packed || !verdict || n < 0 || vk_bits < 1 || sig_bits < 1) return LCB_ERR_INVALID;
    if (!host_only(m, {vk_packed, chmsg, chmsg_off, sig_packed, verdict})) return LCB_ERR_INVALID;
    return on_all(m, n, [&](int, lcb_ctx* c, Shard s) {
        const size_t f = (size_t)s.first;
        const std::vector<int64_t> off = rebased(chmsg_off, s);
        return lcb_lm_verify_packed_batch(c, sch, vk_packed + f * 2 * 32 * vk_bits, vk_bits, chmsg + chmsg_off[s.first], off.data(),
                                          sig_packed + f * c->l * 32 * sig_bits, sig_bits, sig_bias, s.count, bd, wt, verdict + f);
    });
}

int lcb_mctx_bklm_aggregate(lcb_mctx* m, const lcb_scheme* sch, const int16_t* sig_sorted, const uint8_t* agmsg,
                            int64_t agmsg_len, int64_t n, int16_t* ag_sig) {
    LCB_RANGE();
    if (!m || !sch || !sig_sorted || !agmsg || !ag_sig || n < 1 || agmsg_len < 0) return LCB_ERR_INVALID;
    if (!host_only(m, {sig_sorted, agmsg, ag_sig})) return LCB_ERR_INVALID;
    lcb_ctx* c0 = m->ctx[0];
    const size_t words = (size_t)c0->l * c0->d;
    std::vector<void*> part(m->ctx.size(), nullptr);
    int st = on_all(m, n, [&](int i, lcb_ctx* c, Shard s) {
        CK(c, cudaSetDevice(c->device));
        CK(c, cudaMalloc(&part[i], words * sizeof(int32_t) * ew(c)));
        const size_t D_ = (size_t)c->d * ew(c);
        const int r = lcb_bklm_aggregate_partial(c, sch, sig_sorted + (size_t)s.first * c->l * D_, nullptr, agmsg, agmsg_len,
                                                 s.first, s.count, static_cast<int32_t*>(part[i]));
        if (r != LCB_OK) return r;
        return lcb_synchronize(c);
    });
    if (st == LCB_OK) st = reduce_partials(m, part, words);
    if (st == LCB_OK) {
        st = lcb_bklm_aggregate_finish(c0, static_cast<const int32_t*>(part[0]), ag_sig);
        if (st != LCB_OK) m->last_error = c0->last_error;
    }
    for (size_t i = 0; i < part.size(); ++i)
        if (part[i]) { cudaSetDevice(m->ctx[i]->device); cudaFree(part[i]); }
    return st;
}

int lcb_mctx_bklm_aggregate_verify(lcb_mctx* m, const lcb_scheme* sch, const uint16_t* vk_ntt_sorted, const uint8_t* chmsg_sorted,
                                   const int64_t* chmsg_off, const uint8_t* agmsg, int64_t agmsg_len, int64_t n,
                                   const int16_t* ag_sig, int ag_cap, int avf_bd, int avf_wt, uint8_t* verdict) {
    LCB_RANGE();
    if (!m || !sch || !vk_ntt_sorted || !chmsg_off || !agmsg || !ag_sig || !verdict || n < 1 || agmsg_len < 0) return LCB_ERR_INVALID;
    if (!host_only(m, {vk_ntt_sorted, chmsg_sorted, chmsg_off, agmsg, ag_sig, verdict})) return LCB_ERR_INVALID;
    lcb_ctx* c0 = m->ctx[0];
    const size_t words = (size_t)c0->d;
    std::vector<void*> part(m->ctx.size(), nullptr);
    int st = on_all(m, n, [&](int i, lcb_ctx* c, Shard s) {
        CK(c, cudaSetDevice(c->device));
        CK(c, cudaMalloc(&part[i], words * sizeof(int32_t) * ew(c)));
        const size_t D_ = (size_t)c->d * ew(c);
        const std::vector<int64_t> off = rebased(chmsg_off, s);
        const int r = lcb_bklm_aggverify_partial(c, sch, vk_ntt_sorted + (size_t)s.first * 2 * D_, chmsg_sorted + chmsg_off[s.first],
                                                 off.data(), nullptr, agmsg, agmsg_len, s.first, s.count,
                                                 static_cast<int32_t*>(part[i]));
        if (r != LCB_OK) return r;
        return lcb_synchronize(c);
    });
    if (st == LCB_OK) st = reduce_partials(m, part, words);
    if (st == LCB_OK) {
        st = lcb_bklm_aggverify_finish(c0, static_cast<const int32_t*>(part[0]), ag_sig, n, ag_cap, avf_bd, avf_wt, verdict);
        if (st != LCB_OK) m->last_error = c0->last_error;
    }
    for (size_t i = 0; i < part.size(); ++i)
        if (part[i]) { cudaSetDevice(m->ctx[i]->device); cudaFree(part[i]); }
    return st;
}

}  // extern "C"
