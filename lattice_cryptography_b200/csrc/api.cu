// api.cu — the C ABI of lcb200 (include/lcb200.h): context, parameter tables, host<->device staging
// and the composition of the sampler / ring kernels into the reference's scheme operations.
// No CPU fallback: without an sm_100 device lcb_ctx_create fails with LCB_ERR_NO_DEVICE.
#include <cstdio>
#include <cstring>
#include <new>
#include <algorithm>
#include <cstdlib>
#include <string>
#include <vector>

#include <nvtx3/nvToolsExt.h>

#include "../../include/lcb200.h"
#include "engine.h"

using namespace lcb;

struct lcb_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    cudaStream_t copy_stream = nullptr;  // H2D of large host inputs, chunk by chunk, under the kernels (lazy)
    int secpar = 0, q = 0, d = 0, l = 0, rou = 0;
    RingCtx ring{};
    bool generic = false;                // d != 256 or q >= 2^16: ring_generic.cu / k_sampler_g instead of the fast kernels
    bool wide = false;                   // q >= 2^16: int32 / uint32 element formats
    GenCtx gen{};
    uint32_t* d_gen_tab = nullptr;       // generic twiddle tables: w, ws, iw, iws [d] each, pw [2d]
    NttTables* d_tab = nullptr;
    uint32_t* d_a_hat = nullptr;
    bool has_key_ch = false;
    std::string last_error;
    int64_t launches = 0;
    uint8_t* idx_scratch = nullptr;      // sampler index parking (grow-only, stream-ordered reuse)
    size_t idx_scratch_bytes = 0;
    uint2* il_scratch = nullptr;         // bit-split copies of the BKLM aggregation message (grow-only)
    size_t il_scratch_bytes = 0;
    uint32_t* d_mod_tab = nullptr;       // decoder modulus tables for m <= 256 (engine.h), made once
    uint32_t* coop_scratch = nullptr;    // digest scratch of the cooperative low-latency sampler (grow-only)
    size_t coop_scratch_bytes = 0;
    // optional per-kernel CUDA-event timing (lcb_profile_*)
    bool profile = false;
    struct Pending { int id; cudaEvent_t a, b; };
    std::vector<Pending> pending;
    double prof_ms[32] = {0};
    int64_t prof_n[32] = {0};
};

namespace {

// NVTX range over one ABI entry point (SURVEY.md section 5): shows up as a named span on the CPU timeline of nsys /
// ncu; header-only NVTX3 resolves to no-ops when no profiler is attached.
struct NvtxRange {
    explicit NvtxRange(const char* name) { nvtxRangePushA(name); }
    ~NvtxRange() { nvtxRangePop(); }
};
#define LCB_RANGE() NvtxRange nvtx_range_(__func__)

thread_local std::string g_create_error;

int fail(lcb_ctx* c, int status, const std::string& what) {
    if (c) c->last_error = what;
    return status;
}

int fail_cuda(lcb_ctx* c, cudaError_t e, const char* what) {
    return fail(c, e == cudaErrorMemoryAllocation ? LCB_ERR_OOM : LCB_ERR_CUDA,
                std::string(what) + ": " + cudaGetErrorString(e));
}

#define CK(c, call)                                              \
    do {                                                         \
        cudaError_t e_ = (call);                                 \
        if (e_ != cudaSuccess) return fail_cuda((c), e_, #call); \
    } while (0)

// host signatures are moved and verified 2^17 triples at a time (0.87 / 1.5 GB per chunk)
constexpr int64_t kPipeChunk = 1 << 17;

enum KernelId { K_SAMPLER = 0, K_SHAKE, K_NTT_FWD, K_NTT_INV, K_POLY_MUL, K_MATVEC, K_SIGN, K_VERIFY, K_ADDSUB,
                K_AGG_COEFS, K_AGG_PARTIAL, K_AGG_FINISH, K_AGGV_PARTIAL, K_AGGV_FINISH, K_PACK, K_UNPACK, K_GROUP_IDS,
                K_AGG_COEFS_SEG, K_AGG_PARTIAL_SEG, K_AGGV_PARTIAL_SEG, K_AGGV_RESIDUES, K_AGGV_LIMITS, K_AGG_FINISH_PACK,
                K_CONTENT_STR, K_CHALLENGE_INPUTS, K_AGGREGATION_INPUTS, K_COUNT };
const char* const kKernelNames[K_COUNT] = {"sampler", "shake256", "ntt_fwd", "ntt_inv", "poly_mul", "matvec", "sign",
                                           "verify", "vec_addsub", "agg_coefs", "agg_partial", "agg_finish",
                                           "aggv_partial", "aggv_finish", "pack", "unpack", "group_ids",
                                           "agg_coefs_seg", "agg_partial_seg", "aggv_partial_seg", "aggv_residues",
                                           "aggv_limits", "agg_finish_pack", "content_str", "challenge_inputs",
                                           "aggregation_inputs"};
static_assert(K_COUNT <= 32, "grow lcb_ctx::prof_ms / prof_n");

// Launch wrapper: counts the launch and, when profiling is on, brackets it with CUDA events on the
// ctx stream (resolved lazily in lcb_profile_read).
template <typename F>
cudaError_t timed(lcb_ctx* c, int id, F&& launch) {
    c->launches += 1;
    if (!c->profile) return launch();
    lcb_ctx::Pending p{id, nullptr, nullptr};
    cudaError_t e;
    if ((e = cudaEventCreate(&p.a)) != cudaSuccess) return e;
    if ((e = cudaEventCreate(&p.b)) != cudaSuccess) return e;
    if ((e = cudaEventRecord(p.a, c->stream)) != cudaSuccess) return e;
    e = launch();
    cudaEventRecord(p.b, c->stream);
    c->pending.push_back(p);
    return e;
}

// Point a sampler launch at the ctx's index scratch, growing it when the batch needs more.
cudaError_t sampler_scratch(lcb_ctx* c, SamplerArgs& a) {
    // a handful of streams: the cooperative kernel (one block per stream, sponge and per-polynomial decoders side by side)
    a.coop_digest = reinterpret_cast<uint32_t*>(1);
    const bool coop = sampler_coop_applies(a, c->ring.num_sms);
    a.coop_digest = nullptr;
    const int64_t slots = coop ? a.n * a.vec_len : a.n;
    const size_t need = sampler_scratch_bytes(slots, a.wt, true);   // sized for 16-bit indices: either kernel may run
    cudaError_t e;
    if (need > c->idx_scratch_bytes) {
        if ((e = cudaStreamSynchronize(c->stream)) != cudaSuccess) return e;
        if (c->idx_scratch) cudaFree(c->idx_scratch);
        c->idx_scratch = nullptr;
        c->idx_scratch_bytes = 0;
        if ((e = cudaMalloc(&c->idx_scratch, need)) != cudaSuccess) return e;
        c->idx_scratch_bytes = need;
    }
    a.idx_scratch = c->idx_scratch;
    a.idx_stride = sampler_stride(slots);
    if (coop) {
        const int64_t bits = (int64_t)a.logd + (int64_t)(a.wt - 1) * a.idx_bits + (int64_t)a.wt * (1 + a.mag_bits) + a.pad_bits;
        const size_t dneed = (size_t)a.n * sampler_coop_digest_words(a.vec_len, (int)(bits / 32)) * sizeof(uint32_t);
        if (dneed > c->coop_scratch_bytes) {
            if ((e = cudaStreamSynchronize(c->stream)) != cudaSuccess) return e;
            if (c->coop_scratch) cudaFree(c->coop_scratch);
            c->coop_scratch = nullptr;
            c->coop_scratch_bytes = 0;
            if ((e = cudaMalloc(&c->coop_scratch, dneed)) != cudaSuccess) return e;
            c->coop_scratch_bytes = dneed;
        }
        a.coop_digest = c->coop_scratch;
    }
    return cudaSuccess;
}

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

// element counts below are in 16-bit units of the narrow formats; a wide context (q >= 2^16) moves 32-bit elements
inline size_t ew(const lcb_ctx* c) { return c->wide ? 2 : 1; }

int ceil_log2(int v) {
    int c = 0;
    while ((1 << c) < v) ++c;
    return c;
}

bool on_device(const void* p) {
    cudaPointerAttributes at{};
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    return at.type == cudaMemoryTypeDevice || at.type == cudaMemoryTypeManaged;
}

// Per-call staging of caller buffers: device pointers pass through, host pointers are mirrored in
// stream-ordered device scratch (copied in before the kernels, copied back + synchronised after).
class Staging {
  public:
    explicit Staging(lcb_ctx* c) : c_(c) {}
    ~Staging() {
        // an early error return must not free buffers a chunked copy is still writing
        if (piped_ && c_->copy_stream) cudaStreamSynchronize(c_->copy_stream);
        for (cudaEvent_t e : events_) cudaEventDestroy(e);
        // scratch that held secret material (signing keys, witnesses) is cleared before it goes back to the
        // stream-ordered pool: the pool keeps freed blocks resident (release threshold = max) and would hand the
        // bytes to the next allocation of this process
        for (auto& s : secret_) cudaMemsetAsync(s.first, 0, s.second, c_->stream);
        for (void* p : owned_) cudaFreeAsync(p, c_->stream);
    }
    cudaError_t alloc(void** out, size_t bytes, bool secret = false) {
        *out = nullptr;
        if (bytes == 0) bytes = 16;
        cudaError_t e = cudaMallocAsync(out, bytes, c_->stream);
        if (e == cudaSuccess) {
            owned_.push_back(*out);
            if (secret) secret_.push_back({*out, bytes});
        }
        return e;
    }
    // polynomial data (16-bit elements) is moved with 128-bit loads / cp.async: caller-owned DEVICE
    // buffers must be 16-byte aligned (staged host buffers always are)
    template <typename T>
    static bool misaligned(const T* p) { return sizeof(T) == 2 && (reinterpret_cast<uintptr_t>(p) & 15u) != 0; }
    template <typename T>
    cudaError_t in(const T** dev, const T* p, size_t count, bool secret = false) {
        *dev = p;
        if (p == nullptr || count == 0) return cudaSuccess;
        if (on_device(p)) return misaligned(p) ? cudaErrorMisalignedAddress : cudaSuccess;
        void* d = nullptr;
        cudaError_t e = alloc(&d, count * sizeof(T), secret);
        if (e != cudaSuccess) return e;
        host_touched_ = true;
        *dev = static_cast<const T*>(d);
        return cudaMemcpyAsync(d, p, count * sizeof(T), cudaMemcpyHostToDevice, c_->stream);
    }
    // Like in(), but a HOST buffer is only given device room: the caller moves it with pipe_chunk(), one
    // chunk at a time on the copy stream, so that the transfer of chunk i+1 runs under the kernels of chunk i.
    template <typename T>
    cudaError_t in_piped(const T** dev, const T* p, size_t count, bool* piped) {
        *piped = false;
        if (p == nullptr || count == 0 || on_device(p)) return in(dev, p, count);
        void* d = nullptr;
        cudaError_t e = alloc(&d, count * sizeof(T));
        if (e != cudaSuccess) return e;
        host_touched_ = true;
        *dev = static_cast<const T*>(d);
        *piped = true;
        return cudaSuccess;
    }
    // Call once after every allocation of this call and before the first pipe_chunk(): the copy stream may
    // not touch the stream-ordered allocations before the main stream has made them.
    cudaError_t pipe_begin() {
        cudaError_t e;
        if (!c_->copy_stream &&
            (e = cudaStreamCreateWithFlags(&c_->copy_stream, cudaStreamNonBlocking)) != cudaSuccess)
            return e;
        cudaEvent_t ready;
        if ((e = cudaEventCreateWithFlags(&ready, cudaEventDisableTiming)) != cudaSuccess) return e;
        events_.push_back(ready);
        if ((e = cudaEventRecord(ready, c_->stream)) != cudaSuccess) return e;
        piped_ = true;
        return cudaStreamWaitEvent(c_->copy_stream, ready, 0);
    }
    // H2D of one chunk on the copy stream; returns the event the consumer stream has to wait for.
    cudaError_t pipe_chunk(const void* dev, const void* host, size_t bytes, cudaEvent_t* done) {
        cudaError_t e;
        if ((e = cudaEventCreateWithFlags(done, cudaEventDisableTiming)) != cudaSuccess) return e;
        events_.push_back(*done);
        if ((e = cudaMemcpyAsync(const_cast<void*>(dev), host, bytes, cudaMemcpyHostToDevice, c_->copy_stream)) !=
            cudaSuccess)
            return e;
        return cudaEventRecord(*done, c_->copy_stream);
    }
    template <typename T>
    cudaError_t out(T** dev, T* p, size_t count, bool secret = false) {
        *dev = p;
        if (p == nullptr || count == 0) return cudaSuccess;
        if (on_device(p)) return misaligned(p) ? cudaErrorMisalignedAddress : cudaSuccess;
        void* d = nullptr;
        cudaError_t e = alloc(&d, count * sizeof(T), secret);
        if (e != cudaSuccess) return e;
        host_touched_ = true;
        *dev = static_cast<T*>(d);
        back_.push_back({p, d, count * sizeof(T)});
        return cudaSuccess;
    }
    cudaError_t finish() {
        for (auto& b : back_) {
            cudaError_t e = cudaMemcpyAsync(b.host, b.dev, b.bytes, cudaMemcpyDeviceToHost, c_->stream);
            if (e != cudaSuccess) return e;
        }
        back_.clear();
        if (host_touched_) return cudaStreamSynchronize(c_->stream);
        return cudaSuccess;
    }

  private:
    struct Back { void* host; void* dev; size_t bytes; };
    lcb_ctx* c_;
    std::vector<void*> owned_;
    std::vector<std::pair<void*, size_t>> secret_;
    std::vector<Back> back_;
    std::vector<cudaEvent_t> events_;
    bool host_touched_ = false;
    bool piped_ = false;
};

// off[n] = total blob length; needed only to stage a HOST blob, so a device blob costs nothing here
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

std::string salt_of(const char (&s)[LCB_SALT_MAX]) { return std::string(s, strnlen(s, LCB_SALT_MAX)); }

// challenge pairs for n ragged hash inputs (device pointers)
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
        const size_t need = agg_il_bytes(agmsg_len);
        if (need > c->il_scratch_bytes) {
            CK(c, cudaStreamSynchronize(c->stream));
            if (c->il_scratch) cudaFree(c->il_scratch);
            c->il_scratch = nullptr;
            c->il_scratch_bytes = 0;
            CK(c, cudaMalloc(&c->il_scratch, need));
            c->il_scratch_bytes = need;
        }
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
};

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

int group_offsets(lcb_ctx* c, const int64_t* agg_off, const int64_t* agmsg_off, int64_t n_agg, bool nonempty, bool all,
                  GroupOffsets& g) {
    int st = read_offsets(c, agg_off, n_agg, nonempty, all, &g.items, g.agg, "agg_off");
    if (st == LCB_OK) st = read_offsets(c, agmsg_off, n_agg, false, all, &g.msg_bytes, g.msg, "agmsg_off");
    if (st != LCB_OK) return st;
    if (g.items < 0 || g.items > ((int64_t)1 << 30)) return fail(c, LCB_ERR_INVALID, "at most 2^30 signatures per batch call");
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
    const bool fast = !c->generic && sch->ag_wt == 1 && sch->ag_bd == 1;
    if (!fast && (sig_bits || ag_bits)) return fail(c, LCB_ERR_INVALID, "packed aggregation needs monomial coefficients");
    const int l = c->l;
    const size_t D_ = (size_t)c->d * ew(c);
    const size_t pair_len = (size_t)sch->ag_wt * 2 * ew(c);
    int32_t* d_part;
    CK(c, sg.alloc((void**)&d_part, (size_t)n_agg * l * D_ * sizeof(int32_t)));
    CK(c, cudaMemsetAsync(d_part, 0, (size_t)n_agg * l * D_ * sizeof(int32_t), c->stream));
    if (fast) {
        int32_t* d_gid;
        int16_t* d_pairs;
        CK(c, sg.alloc((void**)&d_gid, (size_t)go.items * sizeof(int32_t)));
        CK(c, sg.alloc((void**)&d_pairs, (size_t)go.items * pair_len * sizeof(int16_t)));
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
    int64_t most = 0;
    for (int64_t g = 0; g < n_agg; ++g) most = std::max(most, go.agg[(size_t)g + 1] - go.agg[(size_t)g]);
    int16_t* d_pairs;
    CK(c, sg.alloc((void**)&d_pairs, (size_t)most * pair_len * sizeof(int16_t)));
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
    const bool fast = !c->generic && sch->ag_wt == 1 && sch->ag_bd == 1;
    if (!fast && (vk_bits || ag_bits)) return fail(c, LCB_ERR_INVALID, "packed aggregate verification needs monomial coefficients");
    const int l = c->l;
    const size_t D_ = (size_t)c->d * ew(c);
    const size_t pair_len = (size_t)sch->ag_wt * 2 * ew(c);
    int16_t* d_ch;
    int32_t* d_part;
    CK(c, sg.alloc((void**)&d_ch, (size_t)go.items * sch->ch_wt * 2 * ew(c) * sizeof(int16_t)));
    CK(c, sg.alloc((void**)&d_part, (size_t)n_agg * D_ * sizeof(int32_t)));
    CK(c, cudaMemsetAsync(d_part, 0, (size_t)n_agg * D_ * sizeof(int32_t), c->stream));
    int st;
    if (go.items > 0) {           // the challenges of every item of every group: one sampler launch
        st = run_challenge(c, sch, d_chmsg, d_choff, go.items, d_ch);
        if (st != LCB_OK) return st;
    }
    if (fast) {
        int32_t* d_gid;
        int16_t* d_pairs;
        uint16_t* d_rhs;
        CK(c, sg.alloc((void**)&d_gid, (size_t)go.items * sizeof(int32_t)));
        CK(c, sg.alloc((void**)&d_pairs, (size_t)go.items * pair_len * sizeof(int16_t)));
        CK(c, sg.alloc((void**)&d_rhs, (size_t)n_agg * D * sizeof(uint16_t)));
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
    int64_t most = 0;
    for (int64_t g = 0; g < n_agg; ++g) most = std::max(most, go.agg[(size_t)g + 1] - go.agg[(size_t)g]);
    int16_t* d_pairs;
    CK(c, sg.alloc((void**)&d_pairs, (size_t)most * pair_len * sizeof(int16_t)));
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

// Packed-buffer arguments shared by the packed aggregate calls: widths 1..16, biases 0..32767 (lcb_lm_verify_packed_batch)
bool wire_args_ok(int bits, int bias) { return bits >= 1 && bits <= 16 && bias >= 0 && bias <= 32767; }

}  // namespace

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
    uint32_t psi = 2;
    while (!(powmod(psi, 2 * d, uq) == 1 && powmod(psi, d, uq) != 1)) ++psi;
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
    c->ring.tab = c->d_tab;
    c->ring.a_hat = c->d_a_hat;
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
    const int16_t* d_in;
    CK(c, sg.in(&d_in, key_ch_coef, cnt * ew(c)));
    uint16_t* d_ntt;
    CK(c, sg.alloc((void**)&d_ntt, cnt * ew(c) * sizeof(uint16_t)));
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
    const uint8_t* d_in;
    const int64_t* d_off;
    uint8_t* d_out;
    CK(c, sg.in(&d_in, in, (size_t)total));
    CK(c, sg.in(&d_off, in_off, (size_t)n + 1));
    CK(c, sg.out(&d_out, out, (size_t)(n * out_len)));
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
    uint8_t* d_secret;
    uint8_t* d_out;
    CK(c, sg.alloc((void**)&d_secret, 32, true));           // engine-owned aligned copy, cleared afterwards
    CK(c, cudaMemcpyAsync(d_secret, secret32, 32, cudaMemcpyDefault, c->stream));
    CK(c, sg.out(&d_out, seeds, (size_t)n * c->secpar, true));
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
    CK(c, sg.in(&a.msgs, msgs, (size_t)total));
    CK(c, sg.in(&a.off, msg_off, (size_t)n + 1));
    CK(c, sg.out(&a.out_dense, out_dense, (size_t)n * vec_len * c->d * ew(c)));
    CK(c, sg.out(&a.out_pairs, out_pairs, (size_t)n * vec_len * wt * 2 * ew(c)));
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
    const int16_t* d_in;
    uint16_t* d_out;
    CK(c, sg.in(&d_in, coef, (size_t)npoly * c->d * ew(c)));
    CK(c, sg.out(&d_out, ntt, (size_t)npoly * c->d * ew(c)));
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
    const int16_t* d_in;
    int16_t* d_out;
    CK(c, sg.in(&d_in, coef, (size_t)npoly * c->d * ew(c)));
    CK(c, sg.out(&d_out, rep, (size_t)npoly * 2 * c->d * ew(c)));
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
    const uint16_t* d_in;
    int16_t* d_out;
    CK(c, sg.in(&d_in, ntt, (size_t)npoly * c->d * ew(c)));
    CK(c, sg.out(&d_out, coef, (size_t)npoly * c->d * ew(c)));
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
    const int16_t *d_a, *d_b;
    int16_t* d_out;
    CK(c, sg.in(&d_a, a, (size_t)npoly * c->d * ew(c)));
    CK(c, sg.in(&d_b, b, (size_t)npoly * c->d * ew(c)));
    CK(c, sg.out(&d_out, out, (size_t)npoly * c->d * ew(c)));
    CK(c, timed(c, K_POLY_MUL, [&] {
        return c->generic ? g_launch_poly_mul(c->gen, d_a, d_b, npoly, d_out, c->stream) : launch_poly_mul(c->ring, d_a, d_b, npoly, d_out, c->stream);
    }));
    CK(c, sg.finish());
    return LCB_OK;
}

}  // extern "C"

namespace {

// Packed outputs of lcb_lm_keygen_packed_batch: each chunk's int16 signing keys and uint16 verification keys are packed
// before the next chunk reuses the scratch.  sk / vk may each be null.
struct KeyPack {
    int sk_bits, sk_bias;
    uint8_t *sk, *sk_range;
    int vk_bits;
    uint8_t* vk;
};

// The body of lcb_lm_keygen_batch (pk == null) and of lcb_lm_keygen_packed_batch (pk set, every unpacked output null).
int keygen(lcb_ctx* c, const lcb_scheme* sch, const uint8_t* seeds, const int64_t* seed_off, int64_t n, int16_t* sk_coef,
           uint16_t* sk_ntt, uint16_t* vk_ntt, int16_t* vk_coef, const KeyPack* pk, const char* name) {
    if (!c->has_key_ch) return fail(c, LCB_ERR_NO_KEY_CH, std::string(name) + " before lcb_set_key_ch");
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
    const uint8_t* d_seeds;
    const int64_t* d_off;
    int16_t *d_sk_coef, *d_vk_coef;
    uint16_t *d_sk_ntt, *d_vk_ntt;
    CK(c, sg.in(&d_seeds, seeds, (size_t)total));
    CK(c, sg.in(&d_off, seed_off, (size_t)n + 1));
    const size_t D_ = (size_t)c->d * ew(c);       // 16-bit units per polynomial (twice the degree in a wide context)
    CK(c, sg.out(&d_sk_coef, sk_coef, (size_t)n * 2 * l * D_, true));
    CK(c, sg.out(&d_sk_ntt, sk_ntt, (size_t)n * 2 * l * D_, true));
    CK(c, sg.out(&d_vk_ntt, vk_ntt, (size_t)n * 2 * D_));
    CK(c, sg.out(&d_vk_coef, vk_coef, (size_t)n * 2 * D_));
    uint8_t *d_skp = nullptr, *d_skr = nullptr, *d_vkp = nullptr;
    if (pk) {
        CK(c, sg.out(&d_skp, pk->sk, (size_t)n * 2 * l * 32 * pk->sk_bits, true));
        CK(c, sg.out(&d_skr, pk->sk_range, (size_t)n * 2 * l));
        CK(c, sg.out(&d_vkp, pk->vk, (size_t)n * 2 * 32 * pk->vk_bits));
        if ((reinterpret_cast<uintptr_t>(d_skp) | reinterpret_cast<uintptr_t>(d_vkp)) & 3u)
            return fail(c, LCB_ERR_INVALID, "packed buffers must be 4-byte aligned");
    }
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
    int16_t* scratch = nullptr;
    if (!d_sk_coef) CK(c, sg.alloc((void**)&scratch, (size_t)chunk * 2 * l * D_ * sizeof(int16_t), true));
    uint16_t* vk_scratch = nullptr;                                // NTT-form verification keys of a chunk, to be packed
    if (d_vkp) CK(c, sg.alloc((void**)&vk_scratch, (size_t)chunk * 2 * D_ * sizeof(uint16_t)));
    for (int64_t start = 0; start < n; start += chunk) {
        const int64_t cnt = (n - start < chunk) ? n - start : chunk;
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
                return launch_pack(c->ring, skc, cnt * 2 * l, pk->sk_bits, pk->sk_bias, d_skp + start * 2 * l * 32 * pk->sk_bits,
                                   d_skr ? d_skr + start * 2 * l : nullptr, c->stream);
            }));
        if (d_vkp)
            CK(c, timed(c, K_PACK, [&] {
                return launch_pack(c->ring, vk_scratch, cnt * 2, pk->vk_bits, 0, d_vkp + start * 2 * 32 * pk->vk_bits, nullptr,
                                   c->stream);
            }));
    }
    CK(c, sg.finish());
    return LCB_OK;
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
    if (c->generic) return fail(c, LCB_ERR_INVALID, "the packed wire format is defined for d == 256, q < 2^16 contexts only");
    if (n > ((int64_t)1 << 30)) return fail(c, LCB_ERR_INVALID, "more than 2^30 items in one keygen call");
    const KeyPack pk{sk_bits, sk_bias, sk_packed, sk_packed ? sk_in_range : nullptr, vk_bits, vk_packed};
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
    const uint8_t* d_msg;
    const int64_t* d_off;
    int16_t* d_pairs;
    CK(c, sg.in(&d_msg, chmsg, (size_t)total));
    CK(c, sg.in(&d_off, chmsg_off, (size_t)n + 1));
    CK(c, sg.out(&d_pairs, out_pairs, (size_t)n * sch->ch_wt * 2 * ew(c)));
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
    Staging sg(c);
    const uint16_t* d_sk;
    const uint8_t* d_msg;
    const int64_t* d_off;
    int16_t *d_sig, *d_pairs;
    const size_t D_ = (size_t)c->d * ew(c);
    CK(c, sg.in(&d_sk, sk_ntt, (size_t)n * 2 * l * D_, true));
    CK(c, sg.in(&d_msg, chmsg, (size_t)total));
    CK(c, sg.in(&d_off, chmsg_off, (size_t)n + 1));
    CK(c, sg.out(&d_sig, sig, (size_t)n * l * D_));
    CK(c, sg.alloc((void**)&d_pairs, (size_t)n * sch->ch_wt * 2 * ew(c) * sizeof(int16_t)));
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
    if (!c->has_key_ch) return fail(c, LCB_ERR_NO_KEY_CH, "lcb_lm_verify_batch before lcb_set_key_ch");
    if (n > ((int64_t)1 << 30)) return fail(c, LCB_ERR_INVALID, "more than 2^30 items in one verify call");
    if (n == 0) return LCB_OK;
    CK(c, cudaSetDevice(c->device));
    const int l = c->l;
    int64_t total = 0;
    CK(c, last_offset(c, chmsg, chmsg_off, n, &total));
    Staging sg(c);
    const uint16_t *d_vk, *d_st;
    const uint8_t* d_msg;
    const int64_t* d_off;
    const int16_t* d_sig;
    int16_t* d_pairs;
    uint8_t* d_verdict;
    const size_t D_ = (size_t)c->d * ew(c);
    CK(c, sg.in(&d_vk, vk_ntt, (size_t)n * 2 * D_));
    CK(c, sg.in(&d_msg, chmsg, (size_t)total));
    CK(c, sg.in(&d_off, chmsg_off, (size_t)n + 1));
    bool piped = false;
    CK(c, sg.in_piped(&d_sig, sig, (size_t)n * l * D_, &piped));
    CK(c, sg.in(&d_st, st_ntt, (size_t)n * D_));
    CK(c, sg.out(&d_verdict, verdict, (size_t)n));
    CK(c, sg.alloc((void**)&d_pairs, (size_t)n * sch->ch_wt * 2 * ew(c) * sizeof(int16_t)));
    const int vbd = bd > 32767 ? 32767 : bd;
    // Signatures in HOST memory (the bulk of the bytes) cross PCIe in chunks on the copy stream while the
    // sampler and verify kernels of the previous chunk run; everything else is one launch over the batch.
    const int64_t chunk = piped && n > kPipeChunk ? kPipeChunk : n;
    std::vector<cudaEvent_t> arrived;
    if (piped) {
        CK(c, sg.pipe_begin());
        for (int64_t first = 0; first < n; first += chunk) {
            const int64_t m = n - first < chunk ? n - first : chunk;
            cudaEvent_t ev;
            CK(c, sg.pipe_chunk(d_sig + (size_t)first * l * D_, sig + (size_t)first * l * D_,
                                (size_t)m * l * D_ * sizeof(int16_t), &ev));
            arrived.push_back(ev);
        }
    }
    for (int64_t first = 0, k = 0; first < n; first += chunk, ++k) {
        const int64_t m = n - first < chunk ? n - first : chunk;
        int16_t* pairs = d_pairs + (size_t)first * sch->ch_wt * 2 * ew(c);
        int st = run_challenge(c, sch, d_msg, d_off + first, m, pairs);
        if (st != LCB_OK) return st;
        if (piped) CK(c, cudaStreamWaitEvent(c->stream, arrived[k], 0));
        CK(c, timed(c, K_VERIFY, [&] {
            if (c->generic)
                return g_launch_verify(c->gen, d_sig + (size_t)first * l * D_, d_vk + (size_t)first * 2 * D_, pairs, sch->ch_wt,
                                       nullptr, d_st ? d_st + (size_t)first * D_ : nullptr, m, bd, wt, d_verdict + first, c->stream);
            return launch_verify(c->ring, d_sig + (size_t)first * l * D_, d_vk + (size_t)first * 2 * D_, pairs, sch->ch_wt,
                                 nullptr, d_st ? d_st + (size_t)first * D_ : nullptr, m, vbd, wt, d_verdict + first,
                                 c->stream);
        }));
    }
    CK(c, sg.finish());
    return LCB_OK;
}

// ---- wire format (SURVEY 8(f)2) ----------------------------------------------------------------------
int lcb_pack_batch(lcb_ctx* c, const void* values, int64_t npoly, int bits, int bias, uint8_t* packed,
                   uint8_t* in_range) {
    LCB_RANGE();
    if (!c || !values || !packed || npoly < 0 || bits < 1 || bits > 16 || bias < 0 || bias > 65535) return LCB_ERR_INVALID;
    if (c->generic) return fail(c, LCB_ERR_INVALID, "the packed wire format is defined for d == 256, q < 2^16 contexts only");
    if (npoly == 0) return LCB_OK;
    CK(c, cudaSetDevice(c->device));
    Staging sg(c);
    const uint16_t* d_in;
    uint8_t *d_out, *d_ok;
    CK(c, sg.in(&d_in, static_cast<const uint16_t*>(values), (size_t)npoly * D));
    CK(c, sg.out(&d_out, packed, (size_t)npoly * 32 * bits));
    CK(c, sg.out(&d_ok, in_range, (size_t)npoly));
    if (reinterpret_cast<uintptr_t>(d_out) & 3u) return fail(c, LCB_ERR_INVALID, "packed buffer must be 4-byte aligned");
    CK(c, timed(c, K_PACK, [&] { return launch_pack(c->ring, d_in, npoly, bits, bias, d_out, d_ok, c->stream); }));
    CK(c, sg.finish());
    return LCB_OK;
}

int lcb_unpack_batch(lcb_ctx* c, const uint8_t* packed, int64_t npoly, int bits, int bias, void* values) {
    LCB_RANGE();
    if (!c || !values || !packed || npoly < 0 || bits < 1 || bits > 16 || bias < 0 || bias > 65535) return LCB_ERR_INVALID;
    if (c->generic) return fail(c, LCB_ERR_INVALID, "the packed wire format is defined for d == 256, q < 2^16 contexts only");
    if (npoly == 0) return LCB_OK;
    CK(c, cudaSetDevice(c->device));
    Staging sg(c);
    const uint8_t* d_in;
    uint16_t* d_out;
    CK(c, sg.in(&d_in, packed, (size_t)npoly * 32 * bits));
    CK(c, sg.out(&d_out, static_cast<uint16_t*>(values), (size_t)npoly * D));
    if (reinterpret_cast<uintptr_t>(d_in) & 3u) return fail(c, LCB_ERR_INVALID, "packed buffer must be 4-byte aligned");
    CK(c, timed(c, K_UNPACK, [&] { return launch_unpack(c->ring, d_in, npoly, bits, bias, d_out, c->stream); }));
    CK(c, sg.finish());
    return LCB_OK;
}

// ---- content-mode hash inputs (content.cu) -------------------------------------------------------------------
int lcb_content_str_batch(lcb_ctx* c, int kind, const uint8_t* packed, int bits, int64_t n, uint8_t* out) {
    LCB_RANGE();
    if (!c || !packed || !out || n < 0 || (kind != LCB_CONTENT_VK && kind != LCB_CONTENT_ST) || bits < 1 || bits > 16)
        return LCB_ERR_INVALID;
    if (c->generic) return fail(c, LCB_ERR_INVALID, "the packed wire format is defined for d == 256, q < 2^16 contexts only");
    if (n > ((int64_t)1 << 30)) return fail(c, LCB_ERR_INVALID, "more than 2^30 items in one content-string call");
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
    Staging sg(c);
    const uint8_t* d_in;
    uint8_t* d_out;
    const size_t row_bytes = (size_t)32 * bits;
    CK(c, sg.in(&d_in, packed, (size_t)n * rows * row_bytes));
    CK(c, sg.out(&d_out, out, (size_t)n * 57));
    if (reinterpret_cast<uintptr_t>(d_in) & 3u) return fail(c, LCB_ERR_INVALID, "packed buffer must be 4-byte aligned");
    // unpack -> inverse transform into engine scratch, in chunks of the packed keygen's size (four sampler waves)
    const int64_t wave = (int64_t)c->ring.num_sms * 5 * 128;
    const int64_t chunk = n < 4 * wave ? n : 4 * wave;
    uint16_t* d_ntt;
    int16_t* d_coef;
    CK(c, sg.alloc((void**)&d_ntt, (size_t)chunk * rows * D * sizeof(uint16_t)));
    CK(c, sg.alloc((void**)&d_coef, (size_t)chunk * rows * D * sizeof(int16_t)));
    for (int64_t start = 0; start < n; start += chunk) {
        const int64_t cnt = (n - start < chunk) ? n - start : chunk;
        CK(c, timed(c, K_UNPACK, [&] {
            return launch_unpack(c->ring, d_in + (size_t)start * rows * row_bytes, cnt * rows, bits, 0, d_ntt, c->stream);
        }));
        CK(c, timed(c, K_NTT_INV, [&] { return launch_ntt_inv(c->ring, d_ntt, cnt * rows, d_coef, c->stream); }));
        CK(c, timed(c, K_CONTENT_STR, [&] {
            return launch_content_str(c->ring, d_coef, cnt, rows, prefix, head, d_out + (size_t)start * 57, c->stream);
        }));
    }
    CK(c, sg.finish());
    return LCB_OK;
}

}  // extern "C"

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
    CK(c, sg.in(d_msg, msg + first, (size_t)(last - first)));
    *shift = first;
    return LCB_OK;
}

// a single int64 into a caller buffer, host or device
int put_offset(lcb_ctx* c, int64_t* dst, int64_t v) {
    CK(c, cudaMemcpyAsync(dst, &v, sizeof(int64_t), cudaMemcpyDefault, c->stream));
    CK(c, cudaStreamSynchronize(c->stream));
    return LCB_OK;
}

}  // namespace

extern "C" {

int lcb_challenge_inputs_batch(lcb_ctx* c, const uint8_t* st_str, const uint8_t* vk_str, const uint8_t* msg,
                               const int64_t* msg_off, int64_t n, uint8_t* out, int64_t* out_off) {
    LCB_RANGE();
    if (!c || !vk_str || !msg_off || !out || !out_off || n < 0) return LCB_ERR_INVALID;
    if (n > ((int64_t)1 << 30)) return fail(c, LCB_ERR_INVALID, "more than 2^30 items in one challenge-input call");
    CK(c, cudaSetDevice(c->device));
    if (n == 0) return put_offset(c, out_off, 0);
    int64_t first = 0, last = 0, shift = 0;
    int st = offset_ends(c, msg_off, n, &first, &last, "msg_off");
    if (st != LCB_OK) return st;
    const int64_t per = st_str ? 118 : 59;
    const int64_t out_len = (last - first) + n * per;
    Staging sg(c);
    const uint8_t *d_st = nullptr, *d_vk, *d_msg;
    const int64_t* d_off;
    uint8_t* d_out;
    int64_t* d_out_off;
    st = stage_messages(c, sg, msg, first, last, &d_msg, &shift);
    if (st != LCB_OK) return st;
    CK(c, sg.in(&d_vk, vk_str, (size_t)n * 57));
    if (st_str) CK(c, sg.in(&d_st, st_str, (size_t)n * 57));
    CK(c, sg.in(&d_off, msg_off, (size_t)n + 1));
    CK(c, sg.out(&d_out, out, (size_t)out_len));
    CK(c, sg.out(&d_out_off, out_off, (size_t)n + 1));
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
    if (n_agg > ((int64_t)1 << 30)) return fail(c, LCB_ERR_INVALID, "more than 2^30 aggregates in one call");
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
    const uint8_t *d_vk, *d_msg;
    const int64_t *d_agg, *d_moff;
    int64_t *d_ag, *d_ag_out, shift = 0;
    int32_t* d_gid;
    uint8_t* d_out;
    st = stage_messages(c, sg, msg_sorted, h_moff[0], mlast, &d_msg, &shift);
    if (st != LCB_OK) return st;
    CK(c, sg.in(&d_vk, vk_str_sorted, (size_t)total * 57));
    CK(c, sg.in(&d_agg, agg_off, (size_t)n_agg + 1));
    CK(c, sg.in(&d_moff, msg_off, (size_t)total + 1));
    CK(c, sg.alloc((void**)&d_ag, h_ag.size() * sizeof(int64_t)));
    CK(c, cudaMemcpyAsync(d_ag, h_ag.data(), h_ag.size() * sizeof(int64_t), cudaMemcpyHostToDevice, c->stream));
    CK(c, sg.alloc((void**)&d_gid, (size_t)total * sizeof(int32_t)));
    CK(c, sg.out(&d_out, agmsg, (size_t)out_len));
    CK(c, sg.out(&d_ag_out, agmsg_off, h_ag.size()));
    CK(c, cudaMemcpyAsync(d_ag_out, d_ag, h_ag.size() * sizeof(int64_t), cudaMemcpyDeviceToDevice, c->stream));
    CK(c, timed(c, K_GROUP_IDS, [&] { return launch_group_ids(d_agg, n_agg, total, d_gid, c->ring.num_sms, c->stream); }));
    CK(c, timed(c, K_AGGREGATION_INPUTS, [&] {
        return launch_aggregation_inputs(c->ring, d_agg, d_ag, n_agg, d_gid, total, d_vk, d_msg, shift, d_moff, out_len, d_out,
                                         c->stream);
    }));
    CK(c, sg.finish());
    return LCB_OK;
}

}  // extern "C"

namespace {

// lcb_lm_verify_batch on packed verification keys and signatures, and on packed statements when st_packed is set
// (adaptor verify: the statement is added to the right-hand side, as st_ntt is).  The batch is processed in chunks of
// 2^18: challenge sampler -> k_verify reading the packed rows directly (the shipped 11/14- and 13/16-bit packings, with
// statements at the key width), or unpack -> challenge sampler -> k_verify for any other width (unpacked copies
// bounded to ~2 GB of scratch).  The caller has checked the arguments.
int verify_packed(lcb_ctx* c, const lcb_scheme* sch, const uint8_t* vk_packed, int vk_bits, const uint8_t* chmsg,
                  const int64_t* chmsg_off, const uint8_t* sig_packed, int sig_bits, int sig_bias, const uint8_t* st_packed,
                  int st_bits, int64_t n, int bd, int wt, uint8_t* verdict) {
    if (c->generic) return fail(c, LCB_ERR_INVALID, "the packed wire format is defined for d == 256, q < 2^16 contexts only");
    if (!c->has_key_ch)
        return fail(c, LCB_ERR_NO_KEY_CH, std::string(st_packed ? "lcb_adaptor_verify_packed_batch" : "lcb_lm_verify_packed_batch") +
                                              " before lcb_set_key_ch");
    if (n > ((int64_t)1 << 30)) return fail(c, LCB_ERR_INVALID, "more than 2^30 items in one verify call");
    if (n == 0) return LCB_OK;
    CK(c, cudaSetDevice(c->device));
    const int l = c->l;
    int64_t total = 0;
    CK(c, last_offset(c, chmsg, chmsg_off, n, &total));
    Staging sg(c);
    const uint8_t *d_vkp, *d_sigp, *d_msg, *d_stp = nullptr;
    const int64_t* d_off;
    uint8_t* d_verdict;
    CK(c, sg.in(&d_vkp, vk_packed, (size_t)n * 2 * 32 * vk_bits));
    CK(c, sg.in(&d_msg, chmsg, (size_t)total));
    CK(c, sg.in(&d_off, chmsg_off, (size_t)n + 1));
    bool piped = false;
    CK(c, sg.in_piped(&d_sigp, sig_packed, (size_t)n * l * 32 * sig_bits, &piped));
    if (st_packed) CK(c, sg.in(&d_stp, st_packed, (size_t)n * 32 * st_bits));
    CK(c, sg.out(&d_verdict, verdict, (size_t)n));
    if ((reinterpret_cast<uintptr_t>(d_vkp) | reinterpret_cast<uintptr_t>(d_sigp) | reinterpret_cast<uintptr_t>(d_stp)) & 3u)
        return fail(c, LCB_ERR_INVALID, "packed buffers must be 4-byte aligned");
    const int64_t chunk = n < 2 * kPipeChunk ? n : 2 * kPipeChunk;
    // The two shipped packings (11/14 and 13/16 bits) are expanded inside k_verify; any other width is unpacked
    // into scratch first.
    // The fused route streams packed signature rows with 16-byte cp.async and reads 16-bit key slots with 128-bit
    // loads, so it needs 16-byte aligned buffers (staged host buffers always are); a caller-owned device buffer that
    // is only 4-byte aligned takes the unpack-first route instead of raising a sticky misaligned-address fault.
    // Statements are read like key halves: they must have the key width and, at 16 bits, 16-byte aligned rows.
    const bool aligned16 = (reinterpret_cast<uintptr_t>(d_sigp) & 15u) == 0 &&
                           (vk_bits == 14 || (reinterpret_cast<uintptr_t>(d_vkp) & 15u) == 0) &&
                           (!d_stp || vk_bits == 14 || (reinterpret_cast<uintptr_t>(d_stp) & 15u) == 0);
    const bool fused = aligned16 && (!d_stp || st_bits == vk_bits) &&
                       ((sig_bits == 11 && vk_bits == 14) || (sig_bits == 13 && vk_bits == 16));
    uint16_t *d_vk = nullptr, *d_st = nullptr;
    int16_t *d_sig = nullptr, *d_pairs;
    if (!fused) {
        CK(c, sg.alloc((void**)&d_vk, (size_t)chunk * 2 * D * sizeof(uint16_t)));
        CK(c, sg.alloc((void**)&d_sig, (size_t)chunk * l * D * sizeof(int16_t)));
        if (d_stp) CK(c, sg.alloc((void**)&d_st, (size_t)chunk * D * sizeof(uint16_t)));
    }
    CK(c, sg.alloc((void**)&d_pairs, (size_t)chunk * sch->ch_wt * 2 * sizeof(int16_t)));
    // packed signatures in HOST memory cross PCIe chunk by chunk under the kernels of the previous chunk
    std::vector<cudaEvent_t> arrived;
    const size_t sig_row = (size_t)l * 32 * sig_bits;
    if (piped) {
        CK(c, sg.pipe_begin());
        for (int64_t first = 0; first < n; first += chunk) {
            const int64_t m = n - first < chunk ? n - first : chunk;
            cudaEvent_t ev;
            CK(c, sg.pipe_chunk(d_sigp + (size_t)first * sig_row, sig_packed + (size_t)first * sig_row,
                                (size_t)m * sig_row, &ev));
            arrived.push_back(ev);
        }
    }
    for (int64_t first = 0, k = 0; first < n; first += chunk, ++k) {
        const int64_t m = n - first < chunk ? n - first : chunk;
        if (fused) {
            int st = run_challenge(c, sch, d_msg, d_off + first, m, d_pairs);
            if (st != LCB_OK) return st;
            if (piped) CK(c, cudaStreamWaitEvent(c->stream, arrived[k], 0));
            CK(c, timed(c, K_VERIFY, [&] {
                return launch_verify_packed(c->ring, d_sigp + (size_t)first * sig_row, sig_bits, sig_bias,
                                            d_vkp + (size_t)first * 2 * 32 * vk_bits, vk_bits, d_pairs, sch->ch_wt, m,
                                            bd > 32767 ? 32767 : bd, wt, d_verdict + first, c->stream,
                                            d_stp ? d_stp + (size_t)first * 32 * st_bits : nullptr);
            }));
            continue;
        }
        CK(c, timed(c, K_UNPACK, [&] {
            return launch_unpack(c->ring, d_vkp + (size_t)first * 2 * 32 * vk_bits, m * 2, vk_bits, 0, d_vk, c->stream);
        }));
        if (d_stp)
            CK(c, timed(c, K_UNPACK, [&] {
                return launch_unpack(c->ring, d_stp + (size_t)first * 32 * st_bits, m, st_bits, 0, d_st, c->stream);
            }));
        if (piped) CK(c, cudaStreamWaitEvent(c->stream, arrived[k], 0));
        CK(c, timed(c, K_UNPACK, [&] {
            return launch_unpack(c->ring, d_sigp + (size_t)first * l * 32 * sig_bits, m * l, sig_bits, sig_bias, d_sig,
                                 c->stream);
        }));
        int st = run_challenge(c, sch, d_msg, d_off + first, m, d_pairs);
        if (st != LCB_OK) return st;
        CK(c, timed(c, K_VERIFY, [&] {
            return launch_verify(c->ring, d_sig, d_vk, d_pairs, sch->ch_wt, nullptr, d_st, m, bd > 32767 ? 32767 : bd,
                                 wt, d_verdict + first, c->stream);
        }));
    }
    CK(c, sg.finish());
    return LCB_OK;
}

// polynomials per chunk of the composed wire routes (sign, adapt, extract): bounds their int16 scratch
constexpr int64_t kWireChunkPoly = (int64_t)1 << 20;

}  // namespace

extern "C" {

int lcb_lm_verify_packed_batch(lcb_ctx* c, const lcb_scheme* sch, const uint8_t* vk_packed, int vk_bits,
                               const uint8_t* chmsg, const int64_t* chmsg_off, const uint8_t* sig_packed, int sig_bits,
                               int sig_bias, int64_t n, int bd, int wt, uint8_t* verdict) {
    LCB_RANGE();
    if (!c || !sch || !vk_packed || !chmsg_off || !sig_packed || !verdict || n < 0 || bd < 0 || wt < 0 ||
        vk_bits < 1 || vk_bits > 16 || sig_bits < 1 || sig_bits > 16 || sig_bias < 0 || sig_bias > 32767)
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

}  // extern "C"

namespace {

// The body of lcb_lm_sign_packed_batch over device buffers (d_range nullable): lcb_lm_sign_batch -> lcb_pack_batch.  Fused
// route (11- or 13-bit rows, 16-byte aligned): k_sign writes the packed rows and in_range flags itself.  Anything else signs
// into int16 scratch and packs it with k_pack, in chunks.
int sign_packed(lcb_ctx* c, Staging& sg, const lcb_scheme* sch, const uint16_t* d_sk, const uint8_t* d_msg, const int64_t* d_off,
                int64_t n, int sig_bits, int sig_bias, uint8_t* d_sigp, uint8_t* d_range) {
    const int l = c->l;
    const size_t row = (size_t)32 * sig_bits;
    int16_t* d_pairs;
    CK(c, sg.alloc((void**)&d_pairs, (size_t)n * sch->ch_wt * 2 * sizeof(int16_t)));
    int st = run_challenge(c, sch, d_msg, d_off, n, d_pairs);
    if (st != LCB_OK) return st;
    // k_sign stores whole packed rows with 16-byte stores: a caller-owned device buffer that is only 4-byte aligned
    // takes the composed route
    if ((sig_bits == 11 || sig_bits == 13) && (reinterpret_cast<uintptr_t>(d_sigp) & 15u) == 0) {
        CK(c, timed(c, K_SIGN, [&] {
            return launch_sign_packed(c->ring, d_sk, d_pairs, sch->ch_wt, n, sig_bits, sig_bias, d_sigp, d_range, c->stream);
        }));
    } else {
        const int64_t chunk = n < kWireChunkPoly / l ? n : kWireChunkPoly / l;
        int16_t* d_sig;
        CK(c, sg.alloc((void**)&d_sig, (size_t)chunk * l * D * sizeof(int16_t)));
        for (int64_t first = 0; first < n; first += chunk) {
            const int64_t m = n - first < chunk ? n - first : chunk;
            CK(c, timed(c, K_SIGN, [&] {
                return launch_sign(c->ring, d_sk + (size_t)first * 2 * l * D, d_pairs + (size_t)first * sch->ch_wt * 2,
                                   sch->ch_wt, m, d_sig, c->stream);
            }));
            CK(c, timed(c, K_PACK, [&] {
                return launch_pack(c->ring, d_sig, m * l, sig_bits, sig_bias, d_sigp + (size_t)first * l * row,
                                   d_range ? d_range + (size_t)first * l : nullptr, c->stream);
            }));
        }
    }
    return LCB_OK;
}

}  // namespace

extern "C" {

int lcb_lm_sign_packed_batch(lcb_ctx* c, const lcb_scheme* sch, const uint16_t* sk_ntt, const uint8_t* chmsg,
                             const int64_t* chmsg_off, int64_t n, int sig_bits, int sig_bias, uint8_t* sig_packed,
                             uint8_t* in_range) {
    LCB_RANGE();
    if (!c || !sch || !sk_ntt || !chmsg_off || !sig_packed || n < 0 || !wire_args_ok(sig_bits, sig_bias))
        return LCB_ERR_INVALID;
    if (c->generic) return fail(c, LCB_ERR_INVALID, "the packed wire format is defined for d == 256, q < 2^16 contexts only");
    if (n == 0) return LCB_OK;
    CK(c, cudaSetDevice(c->device));
    const int l = c->l;
    int64_t total = 0;
    CK(c, last_offset(c, chmsg, chmsg_off, n, &total));
    Staging sg(c);
    const uint16_t* d_sk;
    const uint8_t* d_msg;
    const int64_t* d_off;
    uint8_t *d_sigp, *d_range;
    const size_t row = (size_t)32 * sig_bits;
    CK(c, sg.in(&d_sk, sk_ntt, (size_t)n * 2 * l * D, true));
    CK(c, sg.in(&d_msg, chmsg, (size_t)total));
    CK(c, sg.in(&d_off, chmsg_off, (size_t)n + 1));
    CK(c, sg.out(&d_sigp, sig_packed, (size_t)n * l * row));
    CK(c, sg.out(&d_range, in_range, (size_t)n * l));
    if (reinterpret_cast<uintptr_t>(d_sigp) & 3u) return fail(c, LCB_ERR_INVALID, "packed buffer must be 4-byte aligned");
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
    if (c->generic) return fail(c, LCB_ERR_INVALID, "the packed wire format is defined for d == 256, q < 2^16 contexts only");
    if (n > ((int64_t)1 << 30)) return fail(c, LCB_ERR_INVALID, "more than 2^30 items in one sign call");
    if (n == 0) return LCB_OK;
    CK(c, cudaSetDevice(c->device));
    const int l = c->l;
    int64_t total = 0;
    CK(c, last_offset(c, chmsg, chmsg_off, n, &total));
    Staging sg(c);
    const uint8_t *d_skp, *d_msg;
    const int64_t* d_off;
    uint8_t *d_sigp, *d_range;
    const size_t sk_item = (size_t)2 * l * 32 * sk_bits, sig_item = (size_t)l * 32 * sig_bits;
    CK(c, sg.in(&d_skp, sk_packed, (size_t)n * sk_item, true));
    CK(c, sg.in(&d_msg, chmsg, (size_t)total));
    CK(c, sg.in(&d_off, chmsg_off, (size_t)n + 1));
    CK(c, sg.out(&d_sigp, sig_packed, (size_t)n * sig_item));
    CK(c, sg.out(&d_range, in_range, (size_t)n * l));
    if ((reinterpret_cast<uintptr_t>(d_skp) | reinterpret_cast<uintptr_t>(d_sigp)) & 3u)
        return fail(c, LCB_ERR_INVALID, "packed buffers must be 4-byte aligned");
    const bool aligned16 = ((reinterpret_cast<uintptr_t>(d_skp) | reinterpret_cast<uintptr_t>(d_sigp)) & 15u) == 0;
    if (aligned16 && sign_sk_fused_applies(sk_bits, sig_bits, sch->ch_bd, sch->ch_wt)) {
        int16_t* d_pairs;
        CK(c, sg.alloc((void**)&d_pairs, (size_t)n * sch->ch_wt * 2 * sizeof(int16_t)));
        int st = run_challenge(c, sch, d_msg, d_off, n, d_pairs);
        if (st != LCB_OK) return st;
        CK(c, timed(c, K_SIGN, [&] {
            return launch_sign_sk_packed(c->ring, d_skp, sk_bits, sk_bias, d_pairs, sch->ch_bd, sch->ch_wt, n, sig_bits, sig_bias,
                                         d_sigp, d_range, c->stream);
        }));
    } else {
        const int64_t chunk = n < kWireChunkPoly / (2 * l) ? n : kWireChunkPoly / (2 * l);
        int16_t* d_coef;
        uint16_t* d_ntt;
        CK(c, sg.alloc((void**)&d_coef, (size_t)chunk * 2 * l * D * sizeof(int16_t), true));
        CK(c, sg.alloc((void**)&d_ntt, (size_t)chunk * 2 * l * D * sizeof(uint16_t), true));
        for (int64_t first = 0; first < n; first += chunk) {
            const int64_t m = n - first < chunk ? n - first : chunk;
            CK(c, timed(c, K_UNPACK, [&] {
                return launch_unpack(c->ring, d_skp + (size_t)first * sk_item, m * 2 * l, sk_bits, sk_bias, d_coef, c->stream);
            }));
            CK(c, timed(c, K_NTT_FWD, [&] { return launch_ntt_fwd(c->ring, d_coef, m * 2 * l, d_ntt, c->stream); }));
            Staging chunk_sg(c);                 // the chunk's challenge pairs and int16 scratch go back to the pool after it
            int st = sign_packed(c, chunk_sg, sch, d_ntt, d_msg, d_off + first, m, sig_bits, sig_bias,
                                 d_sigp + (size_t)first * sig_item, d_range ? d_range + (size_t)first * l : nullptr);
            if (st != LCB_OK) return st;
        }
    }
    CK(c, sg.finish());
    return LCB_OK;
}

int lcb_bklm_agg_coefs(lcb_ctx* c, const lcb_scheme* sch, const uint8_t* agmsg, int64_t agmsg_len, int64_t first,
                       int64_t count, int16_t* out_pairs) {
    LCB_RANGE();
    if (!c || !sch || !agmsg || !out_pairs || agmsg_len < 0 || first < 0 || count < 0) return LCB_ERR_INVALID;
    if (count == 0) return LCB_OK;
    CK(c, cudaSetDevice(c->device));
    Staging sg(c);
    const uint8_t* d_msg;
    int16_t* d_pairs;
    CK(c, sg.in(&d_msg, agmsg, (size_t)agmsg_len));
    CK(c, sg.out(&d_pairs, out_pairs, (size_t)count * sch->ag_wt * 2 * ew(c)));
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
    Staging sg(c);
    const int16_t *d_sig, *d_pairs_in;
    const uint8_t* d_msg;
    int32_t* d_partial;
    const size_t D_ = (size_t)c->d * ew(c);
    const size_t pair_len = (size_t)sch->ag_wt * 2 * ew(c);
    const bool monomial = sch->ag_wt == 1 && sch->ag_bd == 1;
    if (sch->ag_wt < 1 || sch->ag_wt > c->d || sch->ag_bd < 1) return fail(c, LCB_ERR_INVALID, "bad aggregation parameters");
    CK(c, sg.in(&d_sig, sig_sorted, (size_t)count * l * D_));
    CK(c, sg.in(&d_pairs_in, ag_pairs, (size_t)count * pair_len));
    CK(c, sg.out(&d_partial, partial, (size_t)l * c->d * ew(c)));
    CK(c, cudaMemsetAsync(d_partial, 0, (size_t)l * c->d * ew(c) * sizeof(int32_t), c->stream));
    if (count > 0) {
        if (!d_pairs_in) {
            int16_t* d_pairs;
            CK(c, sg.in(&d_msg, agmsg, (size_t)agmsg_len));
            CK(c, sg.alloc((void**)&d_pairs, (size_t)count * pair_len * sizeof(int16_t)));
            int st = run_agg_coefs(c, sch, d_msg, agmsg_len, first, count, d_pairs);
            if (st != LCB_OK) return st;
            d_pairs_in = d_pairs;
        }
        CK(c, timed(c, K_AGG_PARTIAL, [&] {
            if (!monomial) return g_launch_agg_partial_poly(c->gen, d_sig, d_pairs_in, sch->ag_wt, count, d_partial, c->stream);
            return c->generic ? g_launch_agg_partial(c->gen, d_sig, d_pairs_in, count, d_partial, c->stream)
                              : launch_agg_partial(c->ring, d_sig, d_pairs_in, count, d_partial, c->stream);
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
    const int32_t* d_partial;
    int16_t* d_out;
    CK(c, sg.in(&d_partial, partial_sum, (size_t)c->l * c->d * ew(c)));
    CK(c, sg.out(&d_out, ag_sig, (size_t)c->l * c->d * ew(c)));
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
    Staging sg(c);
    int32_t* d_partial;
    const size_t D_ = (size_t)c->d * ew(c);
    const size_t pair_len = (size_t)sch->ag_wt * 2 * ew(c);
    const bool monomial = sch->ag_wt == 1 && sch->ag_bd == 1;
    if (sch->ag_wt < 1 || sch->ag_wt > c->d || sch->ag_bd < 1) return fail(c, LCB_ERR_INVALID, "bad aggregation parameters");
    CK(c, sg.out(&d_partial, partial, (size_t)c->d * ew(c)));
    CK(c, cudaMemsetAsync(d_partial, 0, (size_t)c->d * ew(c) * sizeof(int32_t), c->stream));
    if (count > 0) {
        int64_t total = 0;
        CK(c, last_offset(c, chmsg_sorted, chmsg_off, count, &total));
        const uint16_t* d_vk;
        const uint8_t *d_chmsg, *d_agmsg;
        const int64_t* d_off;
        const int16_t* d_ag;
        int16_t* d_ch;
        CK(c, sg.in(&d_vk, vk_ntt_sorted, (size_t)count * 2 * D_));
        CK(c, sg.in(&d_chmsg, chmsg_sorted, (size_t)total));
        CK(c, sg.in(&d_off, chmsg_off, (size_t)count + 1));
        CK(c, sg.in(&d_ag, ag_pairs, (size_t)count * pair_len));
        CK(c, sg.alloc((void**)&d_ch, (size_t)count * sch->ch_wt * 2 * ew(c) * sizeof(int16_t)));
        int st = run_challenge(c, sch, d_chmsg, d_off, count, d_ch);
        if (st != LCB_OK) return st;
        if (!d_ag) {
            int16_t* d_pairs;
            CK(c, sg.in(&d_agmsg, agmsg, (size_t)agmsg_len));
            CK(c, sg.alloc((void**)&d_pairs, (size_t)count * pair_len * sizeof(int16_t)));
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
    if (!c->has_key_ch) return fail(c, LCB_ERR_NO_KEY_CH, "lcb_bklm_aggverify_finish before lcb_set_key_ch");
    CK(c, cudaSetDevice(c->device));
    Staging sg(c);
    const int32_t* d_partial;
    const int16_t* d_sig;
    uint8_t* d_verdict;
    CK(c, sg.in(&d_partial, partial_sum, (size_t)c->d * ew(c)));
    CK(c, sg.in(&d_sig, ag_sig, (size_t)c->l * c->d * ew(c)));
    CK(c, sg.out(&d_verdict, verdict, 1));
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
    if (sch->ag_wt < 1 || sch->ag_wt > c->d || sch->ag_bd < 1) return fail(c, LCB_ERR_INVALID, "bad aggregation parameters");
    if (n_agg > ((int64_t)1 << 30)) return fail(c, LCB_ERR_INVALID, "more than 2^30 aggregates in one call");
    if (n_agg == 0) return LCB_OK;
    CK(c, cudaSetDevice(c->device));
    const bool fast = !c->generic && sch->ag_wt == 1 && sch->ag_bd == 1;
    GroupOffsets go;
    int st = group_offsets(c, agg_off, agmsg_off, n_agg, true, !fast, go);
    if (st != LCB_OK) return st;
    const int l = c->l;
    const size_t D_ = (size_t)c->d * ew(c);
    Staging sg(c);
    const int16_t* d_sig;
    const uint8_t* d_msg;
    const int64_t *d_aoff, *d_moff;
    int16_t* d_out;
    CK(c, sg.in(&d_sig, sig_sorted, (size_t)go.items * l * D_));
    CK(c, sg.in(&d_msg, agmsg, (size_t)go.msg_bytes));
    CK(c, sg.in(&d_aoff, agg_off, (size_t)n_agg + 1));
    CK(c, sg.in(&d_moff, agmsg_off, (size_t)n_agg + 1));
    CK(c, sg.out(&d_out, ag_sig, (size_t)n_agg * l * D_));
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
    if (sch->ag_wt < 1 || sch->ag_wt > c->d || sch->ag_bd < 1) return fail(c, LCB_ERR_INVALID, "bad aggregation parameters");
    if (!c->has_key_ch) return fail(c, LCB_ERR_NO_KEY_CH, "lcb_bklm_aggregate_verify_batch before lcb_set_key_ch");
    if (n_agg > ((int64_t)1 << 30)) return fail(c, LCB_ERR_INVALID, "more than 2^30 aggregates in one call");
    if (n_agg == 0) return LCB_OK;
    CK(c, cudaSetDevice(c->device));
    const bool fast = !c->generic && sch->ag_wt == 1 && sch->ag_bd == 1;
    GroupOffsets go;
    int st = group_offsets(c, agg_off, agmsg_off, n_agg, false, !fast, go);
    if (st != LCB_OK) return st;
    if (go.items > 0 && (!vk_ntt_sorted || !chmsg_sorted)) return LCB_ERR_INVALID;
    int64_t ch_bytes = 0;
    std::vector<int64_t> unused;
    if (go.items > 0 && !on_device(chmsg_off)) {
        st = read_offsets(c, chmsg_off, go.items, false, false, &ch_bytes, unused, "chmsg_off");
        if (st != LCB_OK) return st;
    }
    if (go.items > 0) CK(c, last_offset(c, chmsg_sorted, chmsg_off, go.items, &ch_bytes));
    const int l = c->l;
    const size_t D_ = (size_t)c->d * ew(c);
    Staging sg(c);
    const uint16_t* d_vk;
    const uint8_t *d_chmsg, *d_msg;
    const int64_t *d_choff, *d_aoff, *d_moff;
    const int16_t* d_ag;
    uint8_t* d_verdict;
    CK(c, sg.in(&d_vk, vk_ntt_sorted, (size_t)go.items * 2 * D_));
    CK(c, sg.in(&d_chmsg, chmsg_sorted, (size_t)ch_bytes));
    CK(c, sg.in(&d_choff, chmsg_off, (size_t)go.items + 1));
    CK(c, sg.in(&d_msg, agmsg, (size_t)go.msg_bytes));
    CK(c, sg.in(&d_aoff, agg_off, (size_t)n_agg + 1));
    CK(c, sg.in(&d_moff, agmsg_off, (size_t)n_agg + 1));
    CK(c, sg.in(&d_ag, ag_sig, (size_t)n_agg * l * D_));
    CK(c, sg.out(&d_verdict, verdict, (size_t)n_agg));
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
    if (c->generic) return fail(c, LCB_ERR_INVALID, "the packed wire format is defined for d == 256, q < 2^16 contexts only");
    if (sch->ag_wt < 1 || sch->ag_wt > c->d || sch->ag_bd < 1) return fail(c, LCB_ERR_INVALID, "bad aggregation parameters");
    if (n_agg > ((int64_t)1 << 30)) return fail(c, LCB_ERR_INVALID, "more than 2^30 aggregates in one call");
    if (n_agg == 0) return LCB_OK;
    CK(c, cudaSetDevice(c->device));
    const bool monomial = sch->ag_wt == 1 && sch->ag_bd == 1;
    GroupOffsets go;
    int st = group_offsets(c, agg_off, agmsg_off, n_agg, true, !monomial, go);
    if (st != LCB_OK) return st;
    const int l = c->l;
    Staging sg(c);
    const uint8_t *d_sigp, *d_msg;
    const int64_t *d_aoff, *d_moff;
    uint8_t *d_agp, *d_range;
    CK(c, sg.in(&d_sigp, sig_packed, (size_t)go.items * l * 32 * sig_bits));
    CK(c, sg.in(&d_msg, agmsg, (size_t)go.msg_bytes));
    CK(c, sg.in(&d_aoff, agg_off, (size_t)n_agg + 1));
    CK(c, sg.in(&d_moff, agmsg_off, (size_t)n_agg + 1));
    CK(c, sg.out(&d_agp, ag_packed, (size_t)n_agg * l * 32 * ag_bits));
    CK(c, sg.out(&d_range, in_range, (size_t)n_agg * l));
    if ((reinterpret_cast<uintptr_t>(d_sigp) | reinterpret_cast<uintptr_t>(d_agp)) & 3u)
        return fail(c, LCB_ERR_INVALID, "packed buffers must be 4-byte aligned");
    // the fused route reads signature rows with 16-byte loads: a caller-owned device buffer that is only 4-byte aligned
    // takes the unpack-first route
    if (monomial && (sig_bits == 11 || sig_bits == 13) && (reinterpret_cast<uintptr_t>(d_sigp) & 15u) == 0) {
        st = aggregate_batch_dev(c, sch, sg, go, n_agg, d_sigp, sig_bits, sig_bias, d_msg, d_aoff, d_moff, d_agp, ag_bits,
                                 ag_bias, d_range);
    } else {
        int16_t *d_sig, *d_ag;
        CK(c, sg.alloc((void**)&d_sig, (size_t)go.items * l * D * sizeof(int16_t)));
        CK(c, sg.alloc((void**)&d_ag, (size_t)n_agg * l * D * sizeof(int16_t)));
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
    if (c->generic) return fail(c, LCB_ERR_INVALID, "the packed wire format is defined for d == 256, q < 2^16 contexts only");
    if (sch->ag_wt < 1 || sch->ag_wt > c->d || sch->ag_bd < 1) return fail(c, LCB_ERR_INVALID, "bad aggregation parameters");
    if (!c->has_key_ch) return fail(c, LCB_ERR_NO_KEY_CH, "lcb_bklm_aggregate_verify_packed_batch before lcb_set_key_ch");
    if (n_agg > ((int64_t)1 << 30)) return fail(c, LCB_ERR_INVALID, "more than 2^30 aggregates in one call");
    if (n_agg == 0) return LCB_OK;
    CK(c, cudaSetDevice(c->device));
    const bool monomial = sch->ag_wt == 1 && sch->ag_bd == 1;
    GroupOffsets go;
    int st = group_offsets(c, agg_off, agmsg_off, n_agg, false, !monomial, go);
    if (st != LCB_OK) return st;
    if (go.items > 0 && (!vk_packed || !chmsg_sorted)) return LCB_ERR_INVALID;
    int64_t ch_bytes = 0;
    std::vector<int64_t> unused;
    if (go.items > 0 && !on_device(chmsg_off)) {
        st = read_offsets(c, chmsg_off, go.items, false, false, &ch_bytes, unused, "chmsg_off");
        if (st != LCB_OK) return st;
    }
    if (go.items > 0) CK(c, last_offset(c, chmsg_sorted, chmsg_off, go.items, &ch_bytes));
    const int l = c->l;
    Staging sg(c);
    const uint8_t *d_vkp, *d_chmsg, *d_msg, *d_agp;
    const int64_t *d_choff, *d_aoff, *d_moff;
    uint8_t* d_verdict;
    CK(c, sg.in(&d_vkp, vk_packed, (size_t)go.items * 2 * 32 * vk_bits));
    CK(c, sg.in(&d_chmsg, chmsg_sorted, (size_t)ch_bytes));
    CK(c, sg.in(&d_choff, chmsg_off, (size_t)go.items + 1));
    CK(c, sg.in(&d_msg, agmsg, (size_t)go.msg_bytes));
    CK(c, sg.in(&d_aoff, agg_off, (size_t)n_agg + 1));
    CK(c, sg.in(&d_moff, agmsg_off, (size_t)n_agg + 1));
    CK(c, sg.in(&d_agp, ag_packed, (size_t)n_agg * l * 32 * ag_bits));
    CK(c, sg.out(&d_verdict, verdict, (size_t)n_agg));
    if ((reinterpret_cast<uintptr_t>(d_vkp) | reinterpret_cast<uintptr_t>(d_agp)) & 3u)
        return fail(c, LCB_ERR_INVALID, "packed buffers must be 4-byte aligned");
    // the fused route stages aggregate rows with 16-byte cp.async and reads 16-bit key rows with 128-bit loads: a
    // caller-owned device buffer that is only 4-byte aligned takes the unpack-first route
    const bool aligned16 = (reinterpret_cast<uintptr_t>(d_agp) & 15u) == 0 &&
                           (vk_bits == 14 || (reinterpret_cast<uintptr_t>(d_vkp) & 15u) == 0);
    if (monomial && aligned16 && (vk_bits == 14 || vk_bits == 16) && (ag_bits == 12 || ag_bits == 14)) {
        st = aggregate_verify_batch_dev(c, sch, sg, go, n_agg, d_vkp, vk_bits == 14 ? 14 : 0, d_chmsg, d_choff, d_msg, d_aoff,
                                        d_moff, d_agp, ag_bits, ag_bias, ag_cap, avf_bd, avf_wt, d_verdict);
    } else {
        uint16_t* d_vk;
        int16_t* d_ag;
        CK(c, sg.alloc((void**)&d_vk, (size_t)go.items * 2 * D * sizeof(uint16_t)));
        CK(c, sg.alloc((void**)&d_ag, (size_t)n_agg * l * D * sizeof(int16_t)));
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

namespace {

// Packed outputs of lcb_adaptor_witgen_packed_batch: each chunk's int16 witnesses and uint16 NTT-form statements are packed
// before the next chunk reuses the scratch.  wit / st may each be null.
struct WitPack {
    int wit_bits, wit_bias;
    uint8_t *wit, *wit_range;
    int st_bits;
    uint8_t* st;
};

// The body of lcb_adaptor_witgen_batch (wp == null: one pass over the whole batch) and of lcb_adaptor_witgen_packed_batch
// (wp set, every unpacked output null: chunks of kWireChunkPoly / l witnesses in secret scratch).
int witgen(lcb_ctx* c, const lcb_scheme* sch, const uint8_t* seeds, const int64_t* seed_off, int64_t n, int16_t* wit_coef,
           uint16_t* st_ntt, int16_t* st_coef, const WitPack* wp, const char* name) {
    if (!c->has_key_ch) return fail(c, LCB_ERR_NO_KEY_CH, std::string(name) + " before lcb_set_key_ch");
    if (n == 0) return LCB_OK;
    CK(c, cudaSetDevice(c->device));
    const int l = c->l;
    SamplerArgs a{};
    int st = fill_sampler(c, a, salt_of(sch->wit_salt).c_str(), nullptr, sch->wit_bd, sch->wit_wt, l);
    if (st != LCB_OK) return fail(c, st, "bad witness parameters");
    int64_t total = 0;
    CK(c, last_offset(c, seeds, seed_off, n, &total));
    Staging sg(c);
    const uint8_t* d_seeds;
    const int64_t* d_off;
    int16_t *d_wit, *d_st_coef;
    uint16_t* d_st_ntt;
    CK(c, sg.in(&d_seeds, seeds, (size_t)total));
    CK(c, sg.in(&d_off, seed_off, (size_t)n + 1));
    const size_t D_ = (size_t)c->d * ew(c);
    CK(c, sg.out(&d_wit, wit_coef, (size_t)n * l * D_, true));
    CK(c, sg.out(&d_st_ntt, st_ntt, (size_t)n * D_));
    CK(c, sg.out(&d_st_coef, st_coef, (size_t)n * D_));
    uint8_t *d_witp = nullptr, *d_witr = nullptr, *d_stp = nullptr;
    if (wp) {
        CK(c, sg.out(&d_witp, wp->wit, (size_t)n * l * 32 * wp->wit_bits, true));
        CK(c, sg.out(&d_witr, wp->wit_range, (size_t)n * l));
        CK(c, sg.out(&d_stp, wp->st, (size_t)n * 32 * wp->st_bits));
        if ((reinterpret_cast<uintptr_t>(d_witp) | reinterpret_cast<uintptr_t>(d_stp)) & 3u)
            return fail(c, LCB_ERR_INVALID, "packed buffers must be 4-byte aligned");
    }
    const int64_t chunk = wp && n > kWireChunkPoly / l ? kWireChunkPoly / l : n;
    int16_t* scratch = nullptr;
    if (!d_wit) CK(c, sg.alloc((void**)&scratch, (size_t)chunk * l * D_ * sizeof(int16_t), true));
    uint16_t* st_scratch = nullptr;                                // NTT-form statements of a chunk, to be packed
    if (d_stp) CK(c, sg.alloc((void**)&st_scratch, (size_t)chunk * D_ * sizeof(uint16_t)));
    for (int64_t start = 0; start < n; start += chunk) {
        const int64_t cnt = (n - start < chunk) ? n - start : chunk;
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
                return launch_pack(c->ring, wit, cnt * l, wp->wit_bits, wp->wit_bias, d_witp + start * l * 32 * wp->wit_bits,
                                   d_witr ? d_witr + start * l : nullptr, c->stream);
            }));
        if (d_stp)
            CK(c, timed(c, K_PACK, [&] {
                return launch_pack(c->ring, st_scratch, cnt, wp->st_bits, 0, d_stp + start * 32 * wp->st_bits, nullptr, c->stream);
            }));
    }
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
    if (c->generic) return fail(c, LCB_ERR_INVALID, "the packed wire format is defined for d == 256, q < 2^16 contexts only");
    if (n > ((int64_t)1 << 30)) return fail(c, LCB_ERR_INVALID, "more than 2^30 items in one witgen call");
    const WitPack wp{wit_bits, wit_bias, wit_packed, wit_packed ? wit_in_range : nullptr, st_bits, st_packed};
    return witgen(c, sch, seeds, seed_off, n, nullptr, nullptr, nullptr, &wp, "lcb_adaptor_witgen_packed_batch");
}

static int vec_addsub(lcb_ctx* c, const int16_t* a, const int16_t* b, int64_t npoly, int sub, int16_t* out) {
    NvtxRange nvtx_range_(sub ? "lcb_vec_sub_batch" : "lcb_vec_add_batch");
    if (!c || !a || !b || !out || npoly < 0) return LCB_ERR_INVALID;
    CK(c, cudaSetDevice(c->device));
    Staging sg(c);
    const int16_t *d_a, *d_b;
    int16_t* d_out;
    CK(c, sg.in(&d_a, a, (size_t)npoly * c->d * ew(c)));
    CK(c, sg.in(&d_b, b, (size_t)npoly * c->d * ew(c)));
    CK(c, sg.out(&d_out, out, (size_t)npoly * c->d * ew(c)));
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

// adapt / extract on the wire format: unpack -> k_vec_addsub -> (pack), in chunks of bounded int16 scratch.  HBM streams of
// a few thousand operations per signature, so they are composed from the existing kernels and exact by construction.
int lcb_adaptor_adapt_packed_batch(lcb_ctx* c, const uint8_t* presig_packed, int presig_bits, int presig_bias,
                                   const int16_t* wit_coef, int64_t npoly, int sig_bits, int sig_bias, uint8_t* sig_packed,
                                   uint8_t* in_range) {
    LCB_RANGE();
    if (!c || !presig_packed || !wit_coef || !sig_packed || npoly < 0 || !wire_args_ok(presig_bits, presig_bias) ||
        !wire_args_ok(sig_bits, sig_bias))
        return LCB_ERR_INVALID;
    if (c->generic) return fail(c, LCB_ERR_INVALID, "the packed wire format is defined for d == 256, q < 2^16 contexts only");
    if (npoly == 0) return LCB_OK;
    CK(c, cudaSetDevice(c->device));
    Staging sg(c);
    const uint8_t* d_prep;
    const int16_t* d_wit;
    uint8_t *d_sigp, *d_range;
    CK(c, sg.in(&d_prep, presig_packed, (size_t)npoly * 32 * presig_bits));
    CK(c, sg.in(&d_wit, wit_coef, (size_t)npoly * D, true));
    CK(c, sg.out(&d_sigp, sig_packed, (size_t)npoly * 32 * sig_bits));
    CK(c, sg.out(&d_range, in_range, (size_t)npoly));
    if ((reinterpret_cast<uintptr_t>(d_prep) | reinterpret_cast<uintptr_t>(d_sigp)) & 3u)
        return fail(c, LCB_ERR_INVALID, "packed buffers must be 4-byte aligned");
    const int64_t chunk = npoly < kWireChunkPoly ? npoly : kWireChunkPoly;
    int16_t *d_pre, *d_sig;
    CK(c, sg.alloc((void**)&d_pre, (size_t)chunk * D * sizeof(int16_t)));
    CK(c, sg.alloc((void**)&d_sig, (size_t)chunk * D * sizeof(int16_t)));
    for (int64_t first = 0; first < npoly; first += chunk) {
        const int64_t m = npoly - first < chunk ? npoly - first : chunk;
        CK(c, timed(c, K_UNPACK, [&] {
            return launch_unpack(c->ring, d_prep + (size_t)first * 32 * presig_bits, m, presig_bits, presig_bias, d_pre,
                                 c->stream);
        }));
        CK(c, timed(c, K_ADDSUB, [&] { return launch_vec_addsub(c->ring, d_pre, d_wit + (size_t)first * D, m * D, 0, d_sig, c->stream); }));
        CK(c, timed(c, K_PACK, [&] {
            return launch_pack(c->ring, d_sig, m, sig_bits, sig_bias, d_sigp + (size_t)first * 32 * sig_bits,
                               d_range ? d_range + first : nullptr, c->stream);
        }));
    }
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
    if (c->generic) return fail(c, LCB_ERR_INVALID, "the packed wire format is defined for d == 256, q < 2^16 contexts only");
    if (npoly == 0) return LCB_OK;
    CK(c, cudaSetDevice(c->device));
    Staging sg(c);
    const uint8_t *d_sigp, *d_prep;
    int16_t* d_wit;
    CK(c, sg.in(&d_sigp, sig_packed, (size_t)npoly * 32 * sig_bits));
    CK(c, sg.in(&d_prep, presig_packed, (size_t)npoly * 32 * presig_bits));
    CK(c, sg.out(&d_wit, wit_coef, (size_t)npoly * D, true));
    if ((reinterpret_cast<uintptr_t>(d_sigp) | reinterpret_cast<uintptr_t>(d_prep)) & 3u)
        return fail(c, LCB_ERR_INVALID, "packed buffers must be 4-byte aligned");
    const int64_t chunk = npoly < kWireChunkPoly ? npoly : kWireChunkPoly;
    int16_t *d_sig, *d_pre;
    CK(c, sg.alloc((void**)&d_sig, (size_t)chunk * D * sizeof(int16_t)));
    CK(c, sg.alloc((void**)&d_pre, (size_t)chunk * D * sizeof(int16_t)));
    for (int64_t first = 0; first < npoly; first += chunk) {
        const int64_t m = npoly - first < chunk ? npoly - first : chunk;
        CK(c, timed(c, K_UNPACK, [&] {
            return launch_unpack(c->ring, d_sigp + (size_t)first * 32 * sig_bits, m, sig_bits, sig_bias, d_sig, c->stream);
        }));
        CK(c, timed(c, K_UNPACK, [&] {
            return launch_unpack(c->ring, d_prep + (size_t)first * 32 * presig_bits, m, presig_bits, presig_bias, d_pre,
                                 c->stream);
        }));
        CK(c, timed(c, K_ADDSUB, [&] { return launch_vec_addsub(c->ring, d_sig, d_pre, m * D, 1, d_wit + (size_t)first * D, c->stream); }));
    }
    CK(c, sg.finish());
    return LCB_OK;
}

int lcb_adaptor_witness_verify_batch(lcb_ctx* c, const int16_t* wit_coef, const uint16_t* st_ntt, int64_t n, int bd,
                                     int wt, uint8_t* verdict) {
    LCB_RANGE();
    if (!c || !wit_coef || !st_ntt || !verdict || n < 0 || bd < 0 || wt < 0) return LCB_ERR_INVALID;
    if (!c->has_key_ch) return fail(c, LCB_ERR_NO_KEY_CH, "lcb_adaptor_witness_verify_batch before lcb_set_key_ch");
    if (n > ((int64_t)1 << 30)) return fail(c, LCB_ERR_INVALID, "more than 2^30 items in one verify call");
    if (n == 0) return LCB_OK;
    CK(c, cudaSetDevice(c->device));
    Staging sg(c);
    const int16_t* d_wit;
    const uint16_t* d_st;
    uint8_t* d_verdict;
    CK(c, sg.in(&d_wit, wit_coef, (size_t)n * c->l * c->d * ew(c)));
    CK(c, sg.in(&d_st, st_ntt, (size_t)n * c->d * ew(c)));
    CK(c, sg.out(&d_verdict, verdict, (size_t)n));
    CK(c, timed(c, K_VERIFY, [&] {
        return c->generic ? g_launch_verify(c->gen, d_wit, nullptr, nullptr, 0, d_st, nullptr, n, bd, wt, d_verdict, c->stream)
                          : launch_verify(c->ring, d_wit, nullptr, nullptr, 0, d_st, nullptr, n, bd > 32767 ? 32767 : bd, wt, d_verdict,
                                          c->stream);
    }));
    CK(c, sg.finish());
    return LCB_OK;
}

// adapt / extract with packed witnesses: unpack both -> k_vec_addsub -> pack in ONE kernel (k_addsub_packed, every width),
// counted under vec_addsub.  a = presig (adapt) or sig (extract), b = wit (adapt) or presig (extract).
static int addsub_packed(lcb_ctx* c, const uint8_t* a, int a_bits, int a_bias, bool a_secret, const uint8_t* b, int b_bits,
                         int b_bias, bool b_secret, int sub, int64_t npoly, int bits, int bias, bool out_secret, uint8_t* out,
                         uint8_t* in_range) {
    if (!c || !a || !b || !out || npoly < 0 || !wire_args_ok(a_bits, a_bias) || !wire_args_ok(b_bits, b_bias) ||
        !wire_args_ok(bits, bias))
        return LCB_ERR_INVALID;
    if (c->generic) return fail(c, LCB_ERR_INVALID, "the packed wire format is defined for d == 256, q < 2^16 contexts only");
    if (npoly == 0) return LCB_OK;
    CK(c, cudaSetDevice(c->device));
    Staging sg(c);
    const uint8_t *d_a, *d_b;
    uint8_t *d_out, *d_range;
    CK(c, sg.in(&d_a, a, (size_t)npoly * 32 * a_bits, a_secret));
    CK(c, sg.in(&d_b, b, (size_t)npoly * 32 * b_bits, b_secret));
    CK(c, sg.out(&d_out, out, (size_t)npoly * 32 * bits, out_secret));
    CK(c, sg.out(&d_range, in_range, (size_t)npoly));
    if ((reinterpret_cast<uintptr_t>(d_a) | reinterpret_cast<uintptr_t>(d_b) | reinterpret_cast<uintptr_t>(d_out)) & 3u)
        return fail(c, LCB_ERR_INVALID, "packed buffers must be 4-byte aligned");
    CK(c, timed(c, K_ADDSUB, [&] {
        return launch_addsub_packed(c->ring, d_a, a_bits, a_bias, d_b, b_bits, b_bias, sub, npoly, bits, bias, d_out, d_range,
                                    c->stream);
    }));
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
    if (c->generic) return fail(c, LCB_ERR_INVALID, "the packed wire format is defined for d == 256, q < 2^16 contexts only");
    if (!c->has_key_ch) return fail(c, LCB_ERR_NO_KEY_CH, "lcb_adaptor_witness_verify_packed_batch before lcb_set_key_ch");
    if (n > ((int64_t)1 << 30)) return fail(c, LCB_ERR_INVALID, "more than 2^30 items in one verify call");
    if (n == 0) return LCB_OK;
    CK(c, cudaSetDevice(c->device));
    const int l = c->l;
    Staging sg(c);
    const uint8_t *d_witp, *d_stp;
    uint8_t* d_verdict;
    const size_t wit_item = (size_t)l * 32 * wit_bits;
    CK(c, sg.in(&d_witp, wit_packed, (size_t)n * wit_item, true));
    CK(c, sg.in(&d_stp, st_packed, (size_t)n * 32 * st_bits));
    CK(c, sg.out(&d_verdict, verdict, (size_t)n));
    if ((reinterpret_cast<uintptr_t>(d_witp) | reinterpret_cast<uintptr_t>(d_stp)) & 3u)
        return fail(c, LCB_ERR_INVALID, "packed buffers must be 4-byte aligned");
    const int bd_k = bd > 32767 ? 32767 : bd;
    // k_verify stages witness rows with 16-byte cp.async and reads 16-bit statement rows with 128-bit loads: a caller-owned
    // device buffer that is only 4-byte aligned takes the composed route
    const bool aligned16 = (reinterpret_cast<uintptr_t>(d_witp) & 15u) == 0 &&
                           (st_bits == 14 || (reinterpret_cast<uintptr_t>(d_stp) & 15u) == 0);
    const bool fused = aligned16 && st_bits == ceil_log2(c->q) &&
                       ((st_bits == 14 && (wit_bits == 2 || wit_bits == 12)) || (st_bits == 16 && (wit_bits == 2 || wit_bits == 14)));
    if (fused) {
        CK(c, timed(c, K_VERIFY, [&] {
            return launch_verify_rhs_packed(c->ring, d_witp, wit_bits, wit_bias, reinterpret_cast<const uint16_t*>(d_stp), n,
                                            bd_k, wt, d_verdict, c->stream, st_bits);
        }));
    } else {
        const int64_t chunk = n < kWireChunkPoly / l ? n : kWireChunkPoly / l;
        int16_t* d_wit;
        uint16_t* d_st;
        CK(c, sg.alloc((void**)&d_wit, (size_t)chunk * l * D * sizeof(int16_t), true));
        CK(c, sg.alloc((void**)&d_st, (size_t)chunk * D * sizeof(uint16_t)));
        for (int64_t first = 0; first < n; first += chunk) {
            const int64_t m = n - first < chunk ? n - first : chunk;
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
        }
    }
    CK(c, sg.finish());
    return LCB_OK;
}


}  // extern "C"

// ================================================================================================================
// Multi-device context (SURVEY.md 8(b): `devices[], ndev`; 8(e)): ONE call shards a host-resident batch over all
// GPUs of the box.  Independent units (keygen / sign / verify) are split into contiguous ranges - the reference's
// distribute_tasks rule, lm_one_time_sigs.py:194-215: the first n % ndev shards are one longer - and run on one
// host thread per device with no data-path communication.  BKLM aggregate / aggregate_verify shard the SORTED
// list, every device reduces its shard to an int32 partial sum in its own memory, the partial sums travel to device
// 0 as peer copies (NVLink when peer access is available) and are added there by a kernel before the finish step.
// One process per GPU with torch.distributed / NCCL (lattice_cryptography_b200/distributed.py, bench.py) remains the
// way to scale across processes; this is the single-process route for C callers.
#include <thread>

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
