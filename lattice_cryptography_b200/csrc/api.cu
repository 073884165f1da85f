// api.cu — the C ABI of lcb200 (include/lcb200.h): context, parameter tables, profiling, the primitive entry points
// and the composition helpers that the scheme operations of api_lm.cu, api_content.cu, api_bklm.cu and api_adaptor.cu
// share (api_internal.h).  The multi-device context is api_mctx.cu.
// No CPU fallback: without an sm_100 device lcb_ctx_create fails with LCB_ERR_NO_DEVICE.
#include <cstdio>
#include <cstdlib>
#include <new>

#include "api_internal.h"

using namespace lcb;
using namespace lcb::abi;

namespace {

thread_local std::string g_create_error;

const char* const kKernelNames[K_COUNT] = {"sampler", "shake256", "ntt_fwd", "ntt_inv", "poly_mul", "matvec", "sign",
                                           "verify", "vec_addsub", "agg_coefs", "agg_partial", "agg_finish",
                                           "aggv_partial", "aggv_finish", "pack", "unpack", "group_ids",
                                           "agg_coefs_seg", "agg_partial_seg", "aggv_partial_seg", "aggv_residues",
                                           "aggv_limits", "agg_finish_pack", "content_str", "challenge_inputs",
                                           "aggregation_inputs", "content_order", "gather_rows", "gather_ragged"};

uint64_t powmod(uint64_t b, uint64_t e, uint64_t q) {
    uint64_t r = 1;
    b %= q;
    while (e) {
        if (e & 1) r = r * b % q;
        b = b * b % q;
        e >>= 1;
    }
    return r;
}

bool is_prime(int v) {
    if (v < 2) return false;
    for (int f = 2; (int64_t)f * f <= v; ++f)
        if (v % f == 0) return false;
    return true;
}

uint32_t bitrev8(uint32_t v) {
    uint32_t r = 0;
    for (int i = 0; i < 8; ++i) r |= ((v >> i) & 1u) << (7 - i);
    return r;
}

uint32_t shoup(uint32_t w, uint32_t q) { return (uint32_t)(((uint64_t)w << 32) / q); }

uint32_t bitrev(uint32_t v, int bits) {
    uint32_t r = 0;
    for (int i = 0; i < bits; ++i) r |= ((v >> i) & 1u) << (bits - 1 - i);
    return r;
}

}  // namespace

namespace lcb {
namespace abi {

bool on_device(const void* p) {
    cudaPointerAttributes at{};
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    return at.type == cudaMemoryTypeDevice || at.type == cudaMemoryTypeManaged;
}

cudaError_t sampler_scratch(lcb_ctx* c, SamplerArgs& a) {
    // a handful of streams: the cooperative kernel (one block per stream, sponge and per-polynomial decoders side by side)
    a.coop_digest = reinterpret_cast<uint32_t*>(1);
    const bool coop = sampler_coop_applies(a, c->ring.num_sms);
    a.coop_digest = nullptr;
    const int64_t slots = coop ? a.n * a.vec_len : a.n;
    // sized for 16-bit indices: either kernel may run
    cudaError_t e = grow(c, c->idx_scratch, c->idx_scratch_bytes, sampler_scratch_bytes(slots, a.wt, true));
    if (e != cudaSuccess) return e;
    a.idx_scratch = c->idx_scratch;
    a.idx_stride = sampler_stride(slots);
    if (coop) {
        const int64_t bits = (int64_t)a.logd + (int64_t)(a.wt - 1) * a.idx_bits + (int64_t)a.wt * (1 + a.mag_bits) + a.pad_bits;
        const size_t dneed = (size_t)a.n * sampler_coop_digest_words(a.vec_len, (int)(bits / 32)) * sizeof(uint32_t);
        if ((e = grow(c, c->coop_scratch, c->coop_scratch_bytes, dneed)) != cudaSuccess) return e;
        a.coop_digest = c->coop_scratch;
    }
    return cudaSuccess;
}

cudaError_t last_offset(lcb_ctx* c, const void* blob, const int64_t* off, int64_t n, int64_t* total) {
    *total = 0;
    if (blob == nullptr || on_device(blob)) return cudaSuccess;
    if (on_device(off)) {
        cudaError_t e = cudaMemcpyAsync(total, off + n, sizeof(int64_t), cudaMemcpyDeviceToHost, c->stream);
        if (e != cudaSuccess) return e;
        return cudaStreamSynchronize(c->stream);
    }
    *total = off[n];
    return cudaSuccess;
}

int fill_sampler(lcb_ctx* c, SamplerArgs& a, const char* salt, const char* suffix, int bd, int wt, int vec_len) {
    if (bd < 1 || (!c->wide && bd > 32767) || wt < 1 || wt > c->d || vec_len < 1) return LCB_ERR_INVALID;
    std::string s = std::string(salt ? salt : "") + (suffix ? suffix : "");
    if ((int)s.size() > SALT_BYTES) return LCB_ERR_INVALID;
    std::memset(a.salt, 0, sizeof(a.salt));
    std::memcpy(a.salt, s.data(), s.size());
    a.salt_len = (int)s.size();
    a.secpar = c->secpar;
    a.bd = bd;
    a.wt = wt;
    a.vec_len = vec_len;
    const int logd = ceil_log2(c->d);
    a.d = c->d;
    a.logd = logd;
    a.wide = c->wide ? 1 : 0;
    a.stream_salts = nullptr;
    a.stream_salt_len = nullptr;
    a.coop_digest = nullptr;
    a.mod_tab = c->d_mod_tab;
    a.idx_bits = logd + c->secpar;
    const int btd = ceil_log2(bd) + 1 + c->secpar;
    a.mag_bits = btd - 1;
    const int64_t bits = (int64_t)logd + (int64_t)(wt - 1) * a.idx_bits + (int64_t)wt * btd;
    a.pad_bits = (int)(8 * ((bits + 7) / 8) - bits);
    a.paired = 0;
    a.salt2_len = 0;
    a.shared_msg = 0;
    a.shared_len = 0;
    a.index_first = 0;
    a.out_dense = nullptr;
    a.dense_stride = 0;
    a.out_pairs = nullptr;
    a.il_msg = nullptr;
    a.il_stride = 0;
    return LCB_OK;
}

int run_challenge(lcb_ctx* c, const lcb_scheme* sch, const uint8_t* d_msg, const int64_t* d_off, int64_t n,
                  int16_t* d_pairs) {
    SamplerArgs a{};
    int st = fill_sampler(c, a, salt_of(sch->ch_salt).c_str(), nullptr, sch->ch_bd, sch->ch_wt, 1);
    if (st != LCB_OK) return fail(c, st, "bad challenge parameters");
    a.msgs = d_msg;
    a.off = d_off;
    a.n = n;
    a.out_pairs = d_pairs;
    CK(c, sampler_scratch(c, a));
    CK(c, timed(c, K_SAMPLER, [&] { return launch_sampler(a, c->stream); }));
    return LCB_OK;
}

int read_offsets(lcb_ctx* c, const int64_t* off, int64_t n, bool strict, bool all, int64_t* last, std::vector<int64_t>& out,
                 const char* what) {
    if (on_device(off)) {
        if (all) {
            out.resize((size_t)n + 1);
            CK(c, cudaMemcpyAsync(out.data(), off, out.size() * sizeof(int64_t), cudaMemcpyDeviceToHost, c->stream));
        } else {
            CK(c, cudaMemcpyAsync(last, off + n, sizeof(int64_t), cudaMemcpyDeviceToHost, c->stream));
        }
        CK(c, cudaStreamSynchronize(c->stream));
        if (all) *last = out[(size_t)n];
        return LCB_OK;
    }
    if (off[0] != 0) return fail(c, LCB_ERR_INVALID, std::string(what) + " must start at 0");
    for (int64_t i = 0; i < n; ++i)
        if (off[i + 1] < off[i] || (strict && off[i + 1] == off[i]))
            return fail(c, LCB_ERR_INVALID, std::string(what) + (strict ? " must increase (every aggregate needs a signature)"
                                                                         : " must not decrease"));
    if (all) out.assign(off, off + n + 1);
    *last = off[n];
    return LCB_OK;
}

}  // namespace abi
}  // namespace lcb

extern "C" {

const char* lcb_strerror(int status) {
    switch (status) {
        case LCB_OK: return "ok";
        case LCB_ERR_INVALID: return "invalid argument or unsupported parameter set";
        case LCB_ERR_CUDA: return "CUDA runtime error";
        case LCB_ERR_NO_DEVICE: return "no sm_100 CUDA device (lcb200 has no CPU fallback)";
        case LCB_ERR_NO_KEY_CH: return "key_ch not set (call lcb_set_key_ch)";
        case LCB_ERR_OOM: return "out of device memory";
        default: return "unknown lcb status";
    }
}

const char* lcb_last_error(const lcb_ctx* ctx) { return ctx ? ctx->last_error.c_str() : g_create_error.c_str(); }

int lcb_version(void) { return 200; }

int lcb_build_is_checked(void) {
#ifdef LCB_CHECKED
    return 1;
#else
    return 0;
#endif
}

namespace {
__global__ void k_check_selftest(int fail) { LCB_CHECK(!fail); }
}  // namespace

int lcb_checked_selftest(lcb_ctx* c) {
    if (!c) return LCB_ERR_INVALID;
    CK(c, cudaSetDevice(c->device));
    k_check_selftest<<<1, 1, 0, c->stream>>>(1);
    CK(c, cudaGetLastError());
    CK(c, cudaStreamSynchronize(c->stream));
    return LCB_OK;
}

int lcb_ctx_create(lcb_ctx** out, int device, int secpar, int q, int d, int l) {
    LCB_RANGE();
    if (!out) return LCB_ERR_INVALID;
    *out = nullptr;
    g_create_error.clear();
    // fields of logd + secpar / 32 + secpar bits must fit the sampler window (MAX_FIELD_BITS)
    if (d < 32 || d > 1024 || (d & (d - 1)) != 0 || l < 1 || l > 64 || secpar < 1 || secpar > 512 || q < 3 || !is_prime(q) ||
        q % (2 * d) != 1) {
        g_create_error = "supported: power-of-two 32 <= d <= 1024, prime q < 2^31 with q % (2 d) == 1, 1 <= l <= 64, "
                         "1 <= secpar <= 512";
        return LCB_ERR_INVALID;
    }
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || device < 0 || device >= ndev) {
        cudaGetLastError();
        g_create_error = "CUDA device not available";
        return LCB_ERR_NO_DEVICE;
    }
    cudaDeviceProp prop{};
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess || prop.major != 10) {
        cudaGetLastError();
        g_create_error = "device is not sm_100 (B200)";
        return LCB_ERR_NO_DEVICE;
    }
    lcb_ctx* c = new (std::nothrow) lcb_ctx();
    if (!c) return LCB_ERR_OOM;
    c->device = device;
    c->secpar = secpar;
    c->q = q;
    c->d = d;
    c->l = l;
    c->wide = q >= 65536;
    c->generic = d != D || c->wide;
    auto bail = [&](cudaError_t e, const char* what) {
        g_create_error = std::string(what) + ": " + cudaGetErrorString(e);
        lcb_ctx_destroy(c);
        return LCB_ERR_CUDA;
    };
    cudaError_t e;
    if ((e = cudaSetDevice(device)) != cudaSuccess) return bail(e, "cudaSetDevice");
    if ((e = cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking)) != cudaSuccess) return bail(e, "cudaStreamCreate");
    c->own_stream = true;
    {   // stream-ordered scratch: keep freed blocks in the pool instead of returning them at every sync
        cudaMemPool_t pool;
        if (cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess) {
            uint64_t keep = UINT64_MAX;
            cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
        }
    }

    // ---- tables: psi = least element of order exactly 2d (LatticeParameters.rou in lattice_algebra)
    const uint32_t uq = (uint32_t)q;
    // The elements of order 2d are the odd powers of any one of them, so the least is found among d candidates instead of
    // by counting up from 2 (tens of millions of steps for q near 2^31 and small d)
    uint32_t root = 0;
    for (uint32_t h = 2; root == 0; ++h) {
        const uint32_t r = (uint32_t)powmod(h, (uq - 1) / (2 * d), uq);
        if (powmod(r, d, uq) == uq - 1) root = r;
    }
    uint32_t psi = root;
    for (uint32_t k = 3, r2 = (uint32_t)powmod(root, 2, uq), x = root; k < 2 * (uint32_t)d; k += 2) {
        x = (uint32_t)((uint64_t)x * r2 % uq);
        if (x < psi) psi = x;
    }
    c->rou = (int)psi;
    {
        // Tables of the generic kernels (ring_generic.cu): zetas in bit-reversed order, their inverses, Shoup
        // companions, psi^e.  Built for EVERY context: the shipped geometry uses them for the operations that have no
        // fast kernel (aggregation with non-monomial coefficients).
        int logd = 0;
        while ((1 << logd) < d) ++logd;
        std::vector<uint32_t> tab((size_t)6 * d);
        uint32_t *w = tab.data(), *ws = w + d, *iw = ws + d, *iws = iw + d, *pw = iws + d;
        for (uint32_t k = 0; k < (uint32_t)d; ++k) {
            w[k] = (uint32_t)powmod(psi, bitrev(k, logd), uq);
            iw[k] = (uint32_t)powmod(w[k], uq - 2, uq);
            ws[k] = shoup(w[k], uq);
            iws[k] = shoup(iw[k], uq);
        }
        for (uint32_t e2 = 0; e2 < 2 * (uint32_t)d; ++e2) pw[e2] = (uint32_t)powmod(psi, e2, uq);
        if ((e = cudaMalloc(&c->d_gen_tab, tab.size() * sizeof(uint32_t))) != cudaSuccess) return bail(e, "cudaMalloc tables");
        if ((e = cudaMemcpy(c->d_gen_tab, tab.data(), tab.size() * sizeof(uint32_t), cudaMemcpyHostToDevice)) != cudaSuccess)
            return bail(e, "cudaMemcpy tables");
        if (c->generic && (e = cudaMalloc(&c->d_a_hat, (size_t)l * d * sizeof(uint32_t))) != cudaSuccess) return bail(e, "cudaMalloc key_ch");
        GenRing& r = c->gen.r;
        r.q = uq;
        r.half = (uq - 1) / 2;
        r.d = d;
        r.logd = logd;
        r.mu64 = (uint64_t)((((unsigned __int128)1) << 64) / uq);
        r.pos_off = (((1ull << 31) + uq - 1) / uq) * uq;
        r.dinv = (uint32_t)powmod((uint32_t)d, uq - 2, uq);
        r.dinv_s = shoup(r.dinv, uq);
        r.w = c->d_gen_tab;
        r.ws = r.w + d;
        r.iw = r.ws + d;
        r.iws = r.iw + d;
        r.pw = r.iws + d;
        c->gen.a_hat = c->d_a_hat;
        c->gen.l = l;
        c->gen.num_sms = prop.multiProcessorCount;
        c->gen.smem_optin = prop.sharedMemPerBlockOptin;
        c->gen.wide = c->wide;
        c->ring.l = l;
        c->ring.num_sms = prop.multiProcessorCount;
    }
    if (c->generic) {
        *out = c;
        return LCB_OK;
    }
    std::vector<NttTables> host(1);
    NttTables& t = host[0];
    for (uint32_t k = 0; k < 256; ++k) {
        uint32_t w = (uint32_t)powmod(psi, bitrev8(k), uq);
        uint32_t iw = (uint32_t)powmod(w, uq - 2, uq);
        t.w[k] = w;
        t.ws[k] = shoup(w, uq);
        t.iw[k] = iw;
        t.iws[k] = shoup(iw, uq);
        t.oddexp[k] = (uint16_t)(2 * bitrev8(k) + 1);
    }
    for (uint32_t k = 0; k < 256; ++k) {      // FP32-assisted forward twiddles (lcb_device.cuh, StageConstF)
        const float wq = (float)((double)t.w[k] / (double)uq);
        t.f_wq[k] = wq;
        t.f_cst[k] = (float)(12582912.0 - 8388608.0 * (double)wq);
        t.f_kw[k] = (uint32_t)((uint64_t)(0x4B400000u + 2u) * uq - (uint64_t)FP_BIAS * t.w[k]);
    }
    for (uint32_t e2 = 0; e2 < 512; ++e2) {
        t.pw[e2] = (uint32_t)powmod(psi, e2, uq);
        t.pws[e2] = shoup(t.pw[e2], uq);
    }
    {
        // FP32-assisted inverse (lcb_device.cuh, ntt_inv_256_fp): twiddle psi^-e as {w, w/q, cst, kw}
        auto fp_entry = [&](uint32_t w) {
            const float wq = (float)((double)w / (double)uq);
            const float cst = (float)(12582912.0 - 8388608.0 * (double)wq);
            const uint32_t kw = (uint32_t)((uint64_t)(0x4B400000u + 2u) * uq - (uint64_t)FP_BIAS * w);
            uint32_t wq_bits, cst_bits;
            std::memcpy(&wq_bits, &wq, 4);
            std::memcpy(&cst_bits, &cst, 4);
            return make_uint4(w, wq_bits, cst_bits, kw);
        };
        auto inv_tw = [&](int half, int j) { return t.pw[(512 - (256 / half) * j % 512) % 512]; };
        const uint32_t dinv = (uint32_t)powmod((uint32_t)d, uq - 2, uq);
        for (int half = 2; half <= 8; half *= 2)
            for (int j = 0; j < half; ++j) {
                const uint4 e4 = fp_entry(inv_tw(half, j));
                const int k = half + j;
                c->ring.iscf.w[k] = e4.x;
                std::memcpy(&c->ring.iscf.wq[k], &e4.y, 4);
                std::memcpy(&c->ring.iscf.cst[k], &e4.z, 4);
                c->ring.iscf.kw[k] = e4.w;
            }
        for (int lane = 0; lane < 16; ++lane) {
            int pos = 0;
            for (int h16 = 1; h16 <= 8; h16 *= 2)
                for (int r = 0; r < h16; ++r) t.inv_lane[lane][pos++] = fp_entry(inv_tw(16 * h16, lane + 16 * r));
            for (int jj = 0; jj < 16; ++jj) {
                const int i = lane + 16 * jj;
                t.inv_lane[lane][pos++] = fp_entry((uint32_t)((uint64_t)t.pw[(512 - i) % 512] * dinv % uq));
            }
        }
    }
    ModQ& m = c->ring.m;
    m.zero = 0;
    m.q = uq;
    m.negq = (uint32_t)(0u - uq);
    m.barrett = 0xFFFFFFFFu / uq;
    m.cq = ((32768u + uq - 1) / uq) * uq;
    m.cq2 = ((65536u + 2 * uq + uq - 1) / uq) * uq;
    m.half = (uq - 1) / 2;
    m.dinv = (uint32_t)powmod((uint32_t)d, uq - 2, uq);
    m.dinv_s = shoup(m.dinv, uq);
    m.q4 = 4 * uq;
    m.in_off = m.cq + 26 * uq + FP_BIAS;
    m.in_off_q4 = m.in_off + m.q4;
    m.bias_mod_q = FP_BIAS % uq;
    m.z1c = (int32_t)t.w[1] > (int32_t)m.half ? (int32_t)t.w[1] - (int32_t)uq : (int32_t)t.w[1];
    m.k1 = (uint32_t)((((1ull << 30) + (1ull << 15) + uq - 1) / uq) * uq);
    {
        uint64_t inv = uq;                                   // Newton: correct to 3 bits, doubled five times
        for (int it = 0; it < 6; ++it) inv *= 2 - (uint64_t)uq * inv;
        m.qinv_lo = (uint32_t)inv;
        m.qinv_hi = (uint32_t)(inv >> 32);
        const uint64_t lim = ~0ull / uq;
        m.dlim_lo = (uint32_t)lim;
        m.dlim_hi = (uint32_t)(lim >> 32);
        m.kq18 = (((1u << 18) + uq - 1) / uq) * uq;
        m.kw0 = (uint32_t)((uint64_t)(0x4B400000u + 2u) * uq);
    }
    for (int k = 0; k < 16; ++k) {
        c->ring.sc.w[k] = t.w[k];
        c->ring.sc.ws[k] = t.ws[k];
        c->ring.sc.iw[k] = t.iw[k];
        c->ring.sc.iws[k] = t.iws[k];
        c->ring.scf.w[k] = t.w[k];
        c->ring.scf.wq[k] = t.f_wq[k];
        c->ring.scf.cst[k] = t.f_cst[k];
        c->ring.scf.kw[k] = t.f_kw[k];
    }
    if ((e = cudaMalloc(&c->d_tab, sizeof(NttTables))) != cudaSuccess) return bail(e, "cudaMalloc tables");
    if ((e = cudaMemcpy(c->d_tab, &t, sizeof(NttTables), cudaMemcpyHostToDevice)) != cudaSuccess) return bail(e, "cudaMemcpy tables");
    if ((e = cudaMalloc(&c->d_a_hat, (size_t)l * D * sizeof(uint32_t))) != cudaSuccess) return bail(e, "cudaMalloc key_ch");
    if ((e = cudaMalloc(&c->d_tc_b, verify_tc_matrix_bytes(l))) != cudaSuccess) return bail(e, "cudaMalloc key_ch matrices");
    c->ring.tab = c->d_tab;
    c->ring.a_hat = c->d_a_hat;
    c->ring.tc_b = c->d_tc_b;
    c->ring.zeta = t.pw[128];
    c->gen.a_hat = c->d_a_hat;
    c->ring.l = l;
    c->ring.num_sms = prop.multiProcessorCount;
    {
        // the sampler's modulus tables (every m <= 256), so that no block computes them (sampler_device.cuh)
        std::vector<uint32_t> mt(SAMPLER_MOD_TABLE_WORDS);
        fill_sampler_mod_table(mt.data());
        if ((e = cudaMalloc(&c->d_mod_tab, mt.size() * sizeof(uint32_t))) != cudaSuccess) return bail(e, "cudaMalloc sampler tables");
        if ((e = cudaMemcpy(c->d_mod_tab, mt.data(), mt.size() * sizeof(uint32_t), cudaMemcpyHostToDevice)) != cudaSuccess)
            return bail(e, "cudaMemcpy sampler tables");
    }
    *out = c;
    return LCB_OK;
}

int lcb_ctx_destroy(lcb_ctx* c) {
    if (!c) return LCB_OK;
    cudaSetDevice(c->device);
    if (c->stream) cudaStreamSynchronize(c->stream);
    if (c->d_tab) cudaFree(c->d_tab);
    if (c->d_gen_tab) cudaFree(c->d_gen_tab);
    if (c->d_a_hat) cudaFree(c->d_a_hat);
    if (c->d_tc_b) cudaFree(c->d_tc_b);
    if (c->idx_scratch) cudaFree(c->idx_scratch);
    if (c->d_mod_tab) cudaFree(c->d_mod_tab);
    if (c->il_scratch) cudaFree(c->il_scratch);
    if (c->coop_scratch) cudaFree(c->coop_scratch);
    if (c->own_stream && c->stream) cudaStreamDestroy(c->stream);
    if (c->copy_stream) {
        cudaStreamSynchronize(c->copy_stream);
        cudaStreamDestroy(c->copy_stream);
    }
    delete c;
    return LCB_OK;
}

int lcb_ctx_set_stream(lcb_ctx* c, void* cuda_stream) {
    if (!c) return LCB_ERR_INVALID;
    CK(c, cudaSetDevice(c->device));
    CK(c, cudaStreamSynchronize(c->stream));
    if (c->own_stream) cudaStreamDestroy(c->stream);
    c->stream = static_cast<cudaStream_t>(cuda_stream);
    c->own_stream = false;
    return LCB_OK;
}

int lcb_synchronize(lcb_ctx* c) {
    if (!c) return LCB_ERR_INVALID;
    CK(c, cudaSetDevice(c->device));
    CK(c, cudaStreamSynchronize(c->stream));
    return LCB_OK;
}

int lcb_ctx_root_of_unity(const lcb_ctx* c) { return c ? c->rou : LCB_ERR_INVALID; }

int64_t lcb_launch_count(const lcb_ctx* c) { return c ? c->launches : 0; }

static int profile_drain(lcb_ctx* c) {
    if (c->pending.empty()) return LCB_OK;
    CK(c, cudaStreamSynchronize(c->stream));
    for (auto& p : c->pending) {
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, p.a, p.b) == cudaSuccess) {
            c->prof_ms[p.id] += ms;
            c->prof_n[p.id] += 1;
        }
        cudaEventDestroy(p.a);
        cudaEventDestroy(p.b);
    }
    c->pending.clear();
    return LCB_OK;
}

int lcb_profile_enable(lcb_ctx* c, int on) {
    if (!c) return LCB_ERR_INVALID;
    CK(c, cudaSetDevice(c->device));
    int st = profile_drain(c);
    c->profile = on != 0;
    return st;
}

int lcb_profile_reset(lcb_ctx* c) {
    if (!c) return LCB_ERR_INVALID;
    CK(c, cudaSetDevice(c->device));
    int st = profile_drain(c);
    for (int i = 0; i < K_COUNT; ++i) { c->prof_ms[i] = 0; c->prof_n[i] = 0; }
    return st;
}

int lcb_profile_read(lcb_ctx* c, const char* kernel, double* total_ms, int64_t* launches) {
    if (!c || !kernel || !total_ms || !launches) return LCB_ERR_INVALID;
    CK(c, cudaSetDevice(c->device));
    int st = profile_drain(c);
    if (st != LCB_OK) return st;
    for (int i = 0; i < K_COUNT; ++i)
        if (std::strcmp(kernel, kKernelNames[i]) == 0) {
            *total_ms = c->prof_ms[i];
            *launches = c->prof_n[i];
            return LCB_OK;
        }
    return fail(c, LCB_ERR_INVALID, std::string("unknown kernel name ") + kernel);
}

int lcb_set_key_ch(lcb_ctx* c, const int16_t* key_ch_coef) {
    LCB_RANGE();
    if (!c || !key_ch_coef) return LCB_ERR_INVALID;
    CK(c, cudaSetDevice(c->device));
    Staging sg(c);
    const size_t cnt = (size_t)c->l * c->d;
    const int16_t* d_in = sg.in(key_ch_coef, cnt * ew(c));
    uint16_t* d_ntt = sg.alloc<uint16_t>(cnt * ew(c));
    CK(c, sg.status());
    if (c->generic) CK(c, timed(c, K_NTT_FWD, [&] { return g_launch_ntt_fwd(c->gen, d_in, c->l, d_ntt, c->stream); }));
    else CK(c, timed(c, K_NTT_FWD, [&] { return launch_ntt_fwd(c->ring, d_in, c->l, d_ntt, c->stream); }));
    if (c->wide) {
        CK(c, cudaMemcpyAsync(c->d_a_hat, d_ntt, cnt * sizeof(uint32_t), cudaMemcpyDeviceToDevice, c->stream));
        CK(c, cudaStreamSynchronize(c->stream));
    } else {
        // widen to uint32 on the host side of the stream (tiny: l*d values, once per parameter set)
        std::vector<uint16_t> h16(cnt);
        CK(c, cudaMemcpyAsync(h16.data(), d_ntt, h16.size() * sizeof(uint16_t), cudaMemcpyDeviceToHost, c->stream));
        CK(c, cudaStreamSynchronize(c->stream));
        std::vector<uint32_t> h32(h16.begin(), h16.end());
        CK(c, cudaMemcpyAsync(c->d_a_hat, h32.data(), h32.size() * sizeof(uint32_t), cudaMemcpyHostToDevice, c->stream));
        if (!c->generic) CK(c, launch_verify_tc_matrix(c->ring, c->stream));
        CK(c, cudaStreamSynchronize(c->stream));
    }
    c->has_key_ch = true;
    CK(c, sg.finish());
    return LCB_OK;
}

int lcb_shake256_batch(lcb_ctx* c, const uint8_t* in, const int64_t* in_off, int64_t n, uint8_t* out,
                       int64_t out_len) {
    LCB_RANGE();
    if (!c || !in_off || !out || n < 0 || out_len < 0) return LCB_ERR_INVALID;
    if (n == 0 || out_len == 0) return LCB_OK;
    CK(c, cudaSetDevice(c->device));
    int64_t total = 0;
    CK(c, last_offset(c, in, in_off, n, &total));
    Staging sg(c);
    const uint8_t* d_in = sg.in(in, (size_t)total);
    const int64_t* d_off = sg.in(in_off, (size_t)n + 1);
    uint8_t* d_out = sg.out(out, (size_t)(n * out_len));
    CK(c, sg.status());
    CK(c, timed(c, K_SHAKE, [&] { return launch_shake256(d_in, d_off, n, d_out, out_len, c->stream); }));
    CK(c, sg.finish());
    return LCB_OK;
}

int lcb_expand_seeds(lcb_ctx* c, const uint8_t* secret32, int64_t first, int64_t n, uint8_t* seeds) {
    LCB_RANGE();
    if (!c || !secret32 || !seeds || n < 0 || first < 0) return LCB_ERR_INVALID;
    if (c->secpar > 512 || (c->secpar & 7)) return fail(c, LCB_ERR_INVALID, "seed expansion needs secpar to be a multiple of 8, at most 512");
    if (n == 0) return LCB_OK;
    CK(c, cudaSetDevice(c->device));
    Staging sg(c);
    uint8_t* d_secret = sg.alloc<uint8_t>(32, true);           // engine-owned aligned copy, cleared afterwards
    uint8_t* d_out = sg.out(seeds, (size_t)n * c->secpar, true);
    CK(c, sg.status());
    CK(c, cudaMemcpyAsync(d_secret, secret32, 32, cudaMemcpyDefault, c->stream));
    CK(c, timed(c, K_SHAKE, [&] { return launch_seed_expand(d_secret, first, n, c->secpar, d_out, c->stream); }));
    CK(c, sg.finish());
    if (!on_device(secret32)) CK(c, cudaStreamSynchronize(c->stream));     // the caller may wipe its copy on return
    return LCB_OK;
}

int lcb_hash2polyvec_batch(lcb_ctx* c, const char* salt, const uint8_t* msgs, const int64_t* msg_off, int64_t n,
                           int bd, int wt, int vec_len, int16_t* out_dense, int16_t* out_pairs) {
    LCB_RANGE();
    if (!c || !msg_off || n < 0) return LCB_ERR_INVALID;
    if (n == 0) return LCB_OK;
    CK(c, cudaSetDevice(c->device));
    SamplerArgs a{};
    int st = fill_sampler(c, a, salt, nullptr, bd, wt, vec_len);
    if (st != LCB_OK) return fail(c, st, "bad sampler parameters");
    int64_t total = 0;
    CK(c, last_offset(c, msgs, msg_off, n, &total));
    Staging sg(c);
    a.msgs = sg.in(msgs, (size_t)total);
    a.off = sg.in(msg_off, (size_t)n + 1);
    a.out_dense = sg.out(out_dense, (size_t)n * vec_len * c->d * ew(c));
    a.out_pairs = sg.out(out_pairs, (size_t)n * vec_len * wt * 2 * ew(c));
    CK(c, sg.status());
    a.n = n;
    a.dense_stride = (int64_t)vec_len * c->d;
    if (a.out_dense && wt < c->d)
        CK(c, cudaMemsetAsync(a.out_dense, 0, (size_t)n * vec_len * c->d * ew(c) * sizeof(int16_t), c->stream));
    CK(c, sampler_scratch(c, a));
    CK(c, timed(c, K_SAMPLER, [&] { return launch_sampler(a, c->stream); }));
    CK(c, sg.finish());
    return LCB_OK;
}

int lcb_ntt_fwd_batch(lcb_ctx* c, const int16_t* coef, int64_t npoly, uint16_t* ntt) {
    LCB_RANGE();
    if (!c || !coef || !ntt || npoly < 0) return LCB_ERR_INVALID;
    CK(c, cudaSetDevice(c->device));
    Staging sg(c);
    const int16_t* d_in = sg.in(coef, (size_t)npoly * c->d * ew(c));
    uint16_t* d_out = sg.out(ntt, (size_t)npoly * c->d * ew(c));
    CK(c, sg.status());
    CK(c, timed(c, K_NTT_FWD, [&] {
        return c->generic ? g_launch_ntt_fwd(c->gen, d_in, npoly, d_out, c->stream) : launch_ntt_fwd(c->ring, d_in, npoly, d_out, c->stream);
    }));
    CK(c, sg.finish());
    return LCB_OK;
}

int lcb_ntt_reference_repr_batch(lcb_ctx* c, const int16_t* coef, int64_t npoly, int16_t* rep) {
    LCB_RANGE();
    if (!c || !coef || !rep || npoly < 0) return LCB_ERR_INVALID;
    CK(c, cudaSetDevice(c->device));
    Staging sg(c);
    const int16_t* d_in = sg.in(coef, (size_t)npoly * c->d * ew(c));
    int16_t* d_out = sg.out(rep, (size_t)npoly * 2 * c->d * ew(c));
    CK(c, sg.status());
    CK(c, timed(c, K_NTT_FWD, [&] {
        return c->generic ? g_launch_ref_repr(c->gen, d_in, npoly, d_out, c->stream) : launch_ntt_ref_repr(c->ring, d_in, npoly, d_out, c->stream);
    }));
    CK(c, sg.finish());
    return LCB_OK;
}

int lcb_ntt_inv_batch(lcb_ctx* c, const uint16_t* ntt, int64_t npoly, int16_t* coef) {
    LCB_RANGE();
    if (!c || !coef || !ntt || npoly < 0) return LCB_ERR_INVALID;
    CK(c, cudaSetDevice(c->device));
    Staging sg(c);
    const uint16_t* d_in = sg.in(ntt, (size_t)npoly * c->d * ew(c));
    int16_t* d_out = sg.out(coef, (size_t)npoly * c->d * ew(c));
    CK(c, sg.status());
    CK(c, timed(c, K_NTT_INV, [&] {
        return c->generic ? g_launch_ntt_inv(c->gen, d_in, npoly, d_out, c->stream) : launch_ntt_inv(c->ring, d_in, npoly, d_out, c->stream);
    }));
    CK(c, sg.finish());
    return LCB_OK;
}

int lcb_poly_mul_batch(lcb_ctx* c, const int16_t* a, const int16_t* b, int64_t npoly, int16_t* out) {
    LCB_RANGE();
    if (!c || !a || !b || !out || npoly < 0) return LCB_ERR_INVALID;
    CK(c, cudaSetDevice(c->device));
    Staging sg(c);
    const int16_t* d_a = sg.in(a, (size_t)npoly * c->d * ew(c));
    const int16_t* d_b = sg.in(b, (size_t)npoly * c->d * ew(c));
    int16_t* d_out = sg.out(out, (size_t)npoly * c->d * ew(c));
    CK(c, sg.status());
    CK(c, timed(c, K_POLY_MUL, [&] {
        return c->generic ? g_launch_poly_mul(c->gen, d_a, d_b, npoly, d_out, c->stream) : launch_poly_mul(c->ring, d_a, d_b, npoly, d_out, c->stream);
    }));
    CK(c, sg.finish());
    return LCB_OK;
}

static int vec_addsub(lcb_ctx* c, const int16_t* a, const int16_t* b, int64_t npoly, int sub, int16_t* out) {
    NvtxRange nvtx_range_(sub ? "lcb_vec_sub_batch" : "lcb_vec_add_batch");
    if (!c || !a || !b || !out || npoly < 0) return LCB_ERR_INVALID;
    CK(c, cudaSetDevice(c->device));
    Staging sg(c);
    const int16_t* d_a = sg.in(a, (size_t)npoly * c->d * ew(c));
    const int16_t* d_b = sg.in(b, (size_t)npoly * c->d * ew(c));
    int16_t* d_out = sg.out(out, (size_t)npoly * c->d * ew(c));
    CK(c, sg.status());
    CK(c, timed(c, K_ADDSUB, [&] {
        return c->generic ? g_launch_vec_addsub(c->gen, d_a, d_b, npoly * c->d, sub, d_out, c->stream)
                          : launch_vec_addsub(c->ring, d_a, d_b, npoly * D, sub, d_out, c->stream);
    }));
    CK(c, sg.finish());
    return LCB_OK;
}

int lcb_vec_add_batch(lcb_ctx* c, const int16_t* a, const int16_t* b, int64_t npoly, int16_t* out) {
    return vec_addsub(c, a, b, npoly, 0, out);
}

int lcb_vec_sub_batch(lcb_ctx* c, const int16_t* a, const int16_t* b, int64_t npoly, int16_t* out) {
    return vec_addsub(c, a, b, npoly, 1, out);
}

// ---- wire format (SURVEY 8(f)2) ----------------------------------------------------------------------
int lcb_pack_batch(lcb_ctx* c, const void* values, int64_t npoly, int bits, int bias, uint8_t* packed,
                   uint8_t* in_range) {
    LCB_RANGE();
    if (!c || !values || !packed || npoly < 0 || bits < 1 || bits > 16 || bias < 0 || bias > 65535) return LCB_ERR_INVALID;
    if (int st = need_wire(c)) return st;
    if (npoly == 0) return LCB_OK;
    CK(c, cudaSetDevice(c->device));
    Staging sg(c);
    const uint16_t* d_in = sg.in(static_cast<const uint16_t*>(values), (size_t)npoly * D);
    uint8_t* d_out = sg.out(packed, (size_t)npoly * 32 * bits);
    uint8_t* d_ok = sg.out(in_range, (size_t)npoly);
    CK(c, sg.status());
    if (int st = need_aligned4(c, {d_out})) return st;
    CK(c, timed(c, K_PACK, [&] { return launch_pack(c->ring, d_in, npoly, bits, bias, d_out, d_ok, c->stream); }));
    CK(c, sg.finish());
    return LCB_OK;
}

int lcb_unpack_batch(lcb_ctx* c, const uint8_t* packed, int64_t npoly, int bits, int bias, void* values) {
    LCB_RANGE();
    if (!c || !values || !packed || npoly < 0 || bits < 1 || bits > 16 || bias < 0 || bias > 65535) return LCB_ERR_INVALID;
    if (int st = need_wire(c)) return st;
    if (npoly == 0) return LCB_OK;
    CK(c, cudaSetDevice(c->device));
    Staging sg(c);
    const uint8_t* d_in = sg.in(packed, (size_t)npoly * 32 * bits);
    uint16_t* d_out = sg.out(static_cast<uint16_t*>(values), (size_t)npoly * D);
    CK(c, sg.status());
    if (int st = need_aligned4(c, {d_in})) return st;
    CK(c, timed(c, K_UNPACK, [&] { return launch_unpack(c->ring, d_in, npoly, bits, bias, d_out, c->stream); }));
    CK(c, sg.finish());
    return LCB_OK;
}

}  // extern "C"
