// api_internal.h — what the host-side files of the C ABI (api*.cu) share: the context, error reporting, launch
// accounting, per-call staging of caller buffers, the entry guards, and the composition helpers api.cu defines.
// Everything here is internal to liblcb200.so: the namespace is hidden, so no helper joins the exported symbols.
#pragma once
#include <algorithm>
#include <cstdint>
#include <cstring>
#include <initializer_list>
#include <string>
#include <utility>
#include <vector>

#include <nvtx3/nvToolsExt.h>

#include "../../include/lcb200.h"
#include "engine.h"

struct lcb_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    cudaStream_t copy_stream = nullptr;  // H2D of large host inputs, chunk by chunk, under the kernels (lazy)
    int secpar = 0, q = 0, d = 0, l = 0, rou = 0;
    lcb::RingCtx ring{};
    bool generic = false;                // d != 256 or q >= 2^16: ring_generic.cu / k_sampler_g instead of the fast kernels
    bool wide = false;                   // q >= 2^16: int32 / uint32 element formats
    lcb::GenCtx gen{};
    uint32_t* d_gen_tab = nullptr;       // generic twiddle tables: w, ws, iw, iws [d] each, pw [2d]
    lcb::NttTables* d_tab = nullptr;
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

namespace lcb {
namespace abi __attribute__((visibility("hidden"))) {

// NVTX range over one ABI entry point (SURVEY.md section 5): shows up as a named span on the CPU timeline of nsys /
// ncu; header-only NVTX3 resolves to no-ops when no profiler is attached.
struct NvtxRange {
    explicit NvtxRange(const char* name) { nvtxRangePushA(name); }
    ~NvtxRange() { nvtxRangePop(); }
};
#define LCB_RANGE() ::lcb::abi::NvtxRange nvtx_range_(__func__)

inline int fail(lcb_ctx* c, int status, const std::string& what) {
    if (c) c->last_error = what;
    return status;
}

inline int fail_cuda(lcb_ctx* c, cudaError_t e, const char* what) {
    return fail(c, e == cudaErrorMemoryAllocation ? LCB_ERR_OOM : LCB_ERR_CUDA, std::string(what) + ": " + cudaGetErrorString(e));
}

#define CK(c, call)                                                         \
    do {                                                                    \
        cudaError_t e_ = (call);                                            \
        if (e_ != cudaSuccess) return ::lcb::abi::fail_cuda((c), e_, #call); \
    } while (0)

enum KernelId { K_SAMPLER = 0, K_SHAKE, K_NTT_FWD, K_NTT_INV, K_POLY_MUL, K_MATVEC, K_SIGN, K_VERIFY, K_ADDSUB,
                K_AGG_COEFS, K_AGG_PARTIAL, K_AGG_FINISH, K_AGGV_PARTIAL, K_AGGV_FINISH, K_PACK, K_UNPACK, K_GROUP_IDS,
                K_AGG_COEFS_SEG, K_AGG_PARTIAL_SEG, K_AGGV_PARTIAL_SEG, K_AGGV_RESIDUES, K_AGGV_LIMITS, K_AGG_FINISH_PACK,
                K_CONTENT_STR, K_CHALLENGE_INPUTS, K_AGGREGATION_INPUTS, K_COUNT };
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

// polynomials per chunk of the composed wire routes (sign, adapt, extract, witness verify): bounds their int16 scratch
constexpr int64_t kWireChunkPoly = (int64_t)1 << 20;

// element counts below are in 16-bit units of the narrow formats; a wide context (q >= 2^16) moves 32-bit elements
inline size_t ew(const lcb_ctx* c) { return c->wide ? 2 : 1; }

inline int ceil_log2(int v) {
    int c = 0;
    while ((1 << c) < v) ++c;
    return c;
}

inline std::string salt_of(const char (&s)[LCB_SALT_MAX]) { return std::string(s, strnlen(s, LCB_SALT_MAX)); }

// Packed-buffer arguments shared by the packed calls: widths 1..16, biases 0..32767
inline bool wire_args_ok(int bits, int bias) { return bits >= 1 && bits <= 16 && bias >= 0 && bias <= 32767; }

// Pointers that are null count as aligned.
inline bool aligned16(std::initializer_list<const void*> ptrs) {
    for (const void* p : ptrs)
        if (reinterpret_cast<uintptr_t>(p) & 15u) return false;
    return true;
}

// fn(first, m, k) for chunk k, the items [first, first + m) of n in chunks of `chunk` (the last one shorter); the
// first status other than LCB_OK that fn returns ends the loop and is returned.
template <typename F>
int for_chunks(int64_t n, int64_t chunk, F&& fn) {
    for (int64_t first = 0, k = 0; first < n; first += chunk, ++k)
        if (const int st = fn(first, std::min(chunk, n - first), k)) return st;
    return LCB_OK;
}

// ---- entry guards: LCB_OK, or the failing status with the message set ----------------------------------------------
inline int need_wire(lcb_ctx* c) {
    return c->generic ? fail(c, LCB_ERR_INVALID, "the packed wire format is defined for d == 256, q < 2^16 contexts only")
                      : LCB_OK;
}

// the verify kernels index items with 32 bits; `what` completes "more than 2^30 "
inline int within_limit(lcb_ctx* c, int64_t n, const char* what) {
    return n > ((int64_t)1 << 30) ? fail(c, LCB_ERR_INVALID, std::string("more than 2^30 ") + what) : LCB_OK;
}

inline int need_key_ch(lcb_ctx* c, const char* name) {
    return c->has_key_ch ? LCB_OK : fail(c, LCB_ERR_NO_KEY_CH, std::string(name) + " before lcb_set_key_ch");
}

inline int agg_params_ok(lcb_ctx* c, const lcb_scheme* sch) {
    return sch->ag_wt < 1 || sch->ag_wt > c->d || sch->ag_bd < 1 ? fail(c, LCB_ERR_INVALID, "bad aggregation parameters")
                                                                 : LCB_OK;
}

// packed rows are read and written as 32-bit words
inline int need_aligned4(lcb_ctx* c, std::initializer_list<const void*> ptrs) {
    for (const void* p : ptrs)
        if (reinterpret_cast<uintptr_t>(p) & 3u) return fail(c, LCB_ERR_INVALID, "packed buffers must be 4-byte aligned");
    return LCB_OK;
}

// Grow-only ctx scratch: a larger size waits for the stream (earlier launches may still read the old buffer) and
// replaces the buffer.
template <typename T>
cudaError_t grow(lcb_ctx* c, T*& p, size_t& bytes, size_t need) {
    if (need <= bytes) return cudaSuccess;
    cudaError_t e;
    if ((e = cudaStreamSynchronize(c->stream)) != cudaSuccess) return e;
    if (p) cudaFree(p);
    p = nullptr;
    bytes = 0;
    if ((e = cudaMalloc(&p, need)) != cudaSuccess) return e;
    bytes = need;
    return cudaSuccess;
}

bool on_device(const void* p);

// Per-call staging of caller buffers: device pointers pass through, host pointers are mirrored in
// stream-ordered device scratch (copied in before the kernels, copied back + synchronised after).
// in / out / alloc / in_piped return the device pointer.  The first failure is kept: every later call does nothing
// and returns nullptr, so a caller stages a block of buffers and checks status() once before it uses any of them.
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
    cudaError_t status() const { return err_; }
    // `count` elements of device scratch, freed (cleared first when secret) when the call returns
    template <typename T>
    T* alloc(size_t count, bool secret = false) {
        if (err_ != cudaSuccess) return nullptr;
        size_t bytes = count * sizeof(T);
        if (bytes == 0) bytes = 16;
        void* d = nullptr;
        if ((err_ = cudaMallocAsync(&d, bytes, c_->stream)) != cudaSuccess) return nullptr;
        owned_.push_back(d);
        if (secret) secret_.push_back({d, bytes});
        return static_cast<T*>(d);
    }
    // polynomial data (16-bit elements) is moved with 128-bit loads / cp.async: caller-owned DEVICE
    // buffers must be 16-byte aligned (staged host buffers always are)
    template <typename T>
    static bool misaligned(const T* p) { return sizeof(T) == 2 && !aligned16({p}); }
    template <typename T>
    const T* in(const T* p, size_t count, bool secret = false) {
        T* d = room(p, count, secret);
        if (d) err_ = cudaMemcpyAsync(d, p, count * sizeof(T), cudaMemcpyHostToDevice, c_->stream);
        return err_ != cudaSuccess ? nullptr : d ? d : p;
    }
    // Like in(), but a HOST buffer of n items of `item` elements is copied on the copy stream in chunks of `chunk`
    // items, so that the copy of chunk k + 1 runs under the kernels of chunk k: arrived[k] is the event the main
    // stream waits for before it reads chunk k.  A device buffer passes through and leaves `arrived` empty.
    template <typename T>
    const T* in_piped(const T* p, int64_t n, size_t item, int64_t chunk, std::vector<cudaEvent_t>& arrived) {
        T* d = room(p, (size_t)n * item, false);
        if (d) err_ = pipe(d, p, n, item * sizeof(T), chunk, arrived);
        return err_ != cudaSuccess ? nullptr : d ? d : p;
    }
    template <typename T>
    T* out(T* p, size_t count, bool secret = false) {
        T* d = room(p, count, secret);
        if (d) back_.push_back({p, d, count * sizeof(T)});
        return err_ != cudaSuccess ? nullptr : d ? d : p;
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
    // Device room for a HOST buffer; nullptr when p is used in place (null, empty or caller device memory) or staging
    // has failed.
    template <typename T>
    T* room(const T* p, size_t count, bool secret) {
        if (err_ != cudaSuccess || p == nullptr || count == 0) return nullptr;
        if (on_device(p)) {
            if (misaligned(p)) err_ = cudaErrorMisalignedAddress;
            return nullptr;
        }
        T* d = alloc<T>(count, secret);
        if (d) host_touched_ = true;
        return d;
    }
    cudaError_t event(cudaEvent_t* e) {
        cudaError_t r = cudaEventCreateWithFlags(e, cudaEventDisableTiming);
        if (r == cudaSuccess) events_.push_back(*e);
        return r;
    }
    cudaError_t pipe(void* dev, const void* host, int64_t n, size_t item_bytes, int64_t chunk, std::vector<cudaEvent_t>& arrived) {
        cudaError_t e;
        if (!c_->copy_stream && (e = cudaStreamCreateWithFlags(&c_->copy_stream, cudaStreamNonBlocking)) != cudaSuccess)
            return e;
        // the copy stream may not touch the stream-ordered allocation before the main stream has made it
        cudaEvent_t ready;
        if ((e = event(&ready)) != cudaSuccess || (e = cudaEventRecord(ready, c_->stream)) != cudaSuccess) return e;
        piped_ = true;
        if ((e = cudaStreamWaitEvent(c_->copy_stream, ready, 0)) != cudaSuccess) return e;
        return static_cast<cudaError_t>(for_chunks(n, chunk, [&](int64_t first, int64_t m, int64_t) {
            cudaEvent_t done;
            cudaError_t r;
            if ((r = event(&done)) != cudaSuccess) return (int)r;
            arrived.push_back(done);
            const size_t at = (size_t)first * item_bytes;
            if ((r = cudaMemcpyAsync(static_cast<char*>(dev) + at, static_cast<const char*>(host) + at, (size_t)m * item_bytes,
                                     cudaMemcpyHostToDevice, c_->copy_stream)) != cudaSuccess)
                return (int)r;
            return (int)cudaEventRecord(done, c_->copy_stream);
        }));
    }

    struct Back { void* host; void* dev; size_t bytes; };
    lcb_ctx* c_;
    std::vector<void*> owned_;
    std::vector<std::pair<void*, size_t>> secret_;
    std::vector<Back> back_;
    std::vector<cudaEvent_t> events_;
    cudaError_t err_ = cudaSuccess;
    bool host_touched_ = false;
    bool piped_ = false;
};

// Packed outputs of the generators (lcb_lm_keygen_packed_batch, lcb_adaptor_witgen_packed_batch): each chunk's int16
// coefficient-form rows (signing keys / witnesses, secret) and uint16 NTT-form rows (verification keys / statements,
// packed with bias 0) are packed before the next chunk reuses the scratch.  rows / pub may each be null.
struct PackedOut {
    int bits, bias;
    uint8_t *rows, *in_range;
    int pub_bits;
    uint8_t* pub;
};

// ---- composition helpers (api.cu) ------------------------------------------------------------------------------------
// Point a sampler launch at the ctx's index scratch, growing it when the batch needs more.
cudaError_t sampler_scratch(lcb_ctx* c, SamplerArgs& a);
int fill_sampler(lcb_ctx* c, SamplerArgs& a, const char* salt, const char* suffix, int bd, int wt, int vec_len);
// challenge pairs for n ragged hash inputs (device pointers)
int run_challenge(lcb_ctx* c, const lcb_scheme* sch, const uint8_t* d_msg, const int64_t* d_off, int64_t n, int16_t* d_pairs);
// off[n] = total blob length; needed only to stage a HOST blob, so a device blob costs nothing here
cudaError_t last_offset(lcb_ctx* c, const void* blob, const int64_t* off, int64_t n, int64_t* total);
// off[n] (and, when `all`, every entry) of an offset array on the host; a host array is checked (starts at 0, never
// decreases; strictly increases when `strict`), a device array is trusted and copied back as far as needed
int read_offsets(lcb_ctx* c, const int64_t* off, int64_t n, bool strict, bool all, int64_t* last, std::vector<int64_t>& out,
                 const char* what);

}  // namespace abi
}  // namespace lcb
