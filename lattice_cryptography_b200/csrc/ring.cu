// ring.cu — polynomial-ring kernels over Z_q[X]/(X^256+1) (sm_100a).
//
// Replaces, batched over independent instances, the reference's arithmetic call sites:
//   key_ch * sk / key_ch * wit          lm_one_time_sigs.py:95-96, adaptor_sigs.py:100     -> k_matvec
//   sk_left ** c + sk_right             lm_one_time_sigs.py:168, adaptor_sigs.py:193       -> k_sign
//   bounds; key_ch*sig == vk0*c+vk1[+st] lm_one_time_sigs.py:173-191, adaptor_sigs.py:198-266 -> k_verify
//                                       (k_verify_tc: int16 rows of large batches, on the tensor cores)
//   sum(sig ** ag)                      bklm_one_time_agg_sigs.py:96                       -> k_agg_partial
//   sum((vk0*c+vk1)*ag); key_ch*ag_sig == . bklm_one_time_agg_sigs.py:99-116               -> k_aggv_*
//   the same for many aggregates per call                                                  -> k_agg*_partial_seg
//   presig + wit, sig - presig          adaptor_sigs.py:221,225                            -> k_vec_addsub
//
// Work mapping: one polynomial vector (one signature / key half / instance) per HALF-WARP; a lane
// holds 16 coefficients; the public row key_ch stays NTT-resident in shared memory (uint32[l][256])
// for the life of the kernel; accumulation of the row-vector product is 64-bit (IMAD.WIDE) with a
// single reduction per output coefficient.  Grids are persistent: (#SM x resident blocks) blocks
// striding over the batch.
#include <cstdlib>

#include "engine.h"
#include "tc_device.cuh"

namespace lcb {

namespace {

constexpr int RBS = 128;                 // threads per block
constexpr int HWB = RBS / LANES;         // half-warps (work items) per block iteration
#ifdef LCB_EXP_MBS
constexpr int MBS = LCB_EXP_MBS;
#else
constexpr int MBS = 512;                 // threads per block of k_matvec: one key_ch copy per SM, as in k_verify (1.89 ->
                                         // 1.78 ms for 2^17 keygen + witgen products)
#endif
constexpr int MHWB = MBS / LANES;

struct HalfWarp {
    int lane;        // 0..15
    int slot;        // half-warp index within the block
    uint32_t* xb;    // transposition buffer of this half-warp
    unsigned mask;   // ballot mask of this half-warp
};

__device__ __forceinline__ HalfWarp half_warp(uint32_t* xbase) {
    const int tid = threadIdx.x;
    HalfWarp h;
    h.lane = tid & 15;
    h.slot = tid >> 4;
    const int upper = (tid >> 4) & 1;
    h.xb = xbase + (tid >> 5) * XWARP + upper * XHALF;
    h.mask = upper ? 0xFFFF0000u : 0x0000FFFFu;
    return h;
}

// coefficient-form polynomial (int16, natural order) -> layout A registers, made non-negative
__device__ __forceinline__ void load_coef_a(uint32_t (&r)[EPT], const int16_t* __restrict__ p, int lane, uint32_t cq) {
#pragma unroll
    for (int j = 0; j < EPT; ++j) r[j] = (uint32_t)((int)__ldg(p + lane + 16 * j) + (int)cq);
}

__device__ __forceinline__ void load_coef_raw(int (&x)[EPT], const int16_t* __restrict__ p, int lane) {
#pragma unroll
    for (int j = 0; j < EPT; ++j) x[j] = (int)__ldg(p + lane + 16 * j);
}

__device__ __forceinline__ void store_coef_a(int16_t* __restrict__ p, const uint32_t (&r)[EPT], int lane, const ModQ& m) {
#pragma unroll
    for (int j = 0; j < EPT; ++j) p[lane + 16 * j] = (int16_t)finish_coef(r[j], m);
}

// key_ch rows in shared memory: the 16 slots of lane t start at word XROW*t (pitch 20, like the
// transposition buffer) so that the 128-bit reads of a quarter-warp fall in 8 distinct bank groups.
constexpr int AROW = LANES * XROW;   // 320 words per row

// sparse (index, coefficient) pairs -> dense polynomial in layout A (via the transposition buffer), as raw signed
// coefficients (input of the FP32-assisted transform)
__device__ __forceinline__ void load_pairs_raw(int (&x)[EPT], const int16_t* __restrict__ pairs, int wt, uint32_t* xb,
                                               int lane) {
#pragma unroll
    for (int j = 0; j < EPT; ++j) xb[XROW * j + lane] = 0;
    __syncwarp();
    const uint32_t* pp = reinterpret_cast<const uint32_t*>(pairs);
    for (int e = lane; e < wt; e += LANES) {
        uint32_t pr = __ldg(pp + e);
        int idx = (int)(pr & 0xFFu);
        xb[XROW * (idx >> 4) + (idx & 15)] = (uint32_t)(int)(int16_t)(pr >> 16);
    }
    __syncwarp();
#pragma unroll
    for (int j = 0; j < EPT; ++j) x[j] = (int)xb[XROW * j + lane];
    __syncwarp();
}

__device__ __forceinline__ void copy_a_hat(uint32_t* dst, const uint32_t* __restrict__ src, int l) {
    const uint4* s4 = reinterpret_cast<const uint4*>(src);
    for (int i = threadIdx.x; i < l * (D / 4); i += blockDim.x) {
        const int row = i >> 6, q4 = i & 63;            // q4: group of 4 slots within the row
        *reinterpret_cast<uint4*>(dst + row * AROW + XROW * (q4 >> 2) + 4 * (q4 & 3)) = __ldg(s4 + i);
    }
    __syncthreads();
}

// acc[m] += r[m] * a_hat_row[slot 16 lane + m]
__device__ __forceinline__ void mac_row(uint64_t (&acc)[EPT], const uint32_t (&r)[EPT], const uint32_t* row, int lane) {
#pragma unroll
    for (int g = 0; g < 4; ++g) {
        uint4 v = *reinterpret_cast<const uint4*>(row + XROW * lane + 4 * g);
        acc[4 * g] += (uint64_t)r[4 * g] * v.x;
        acc[4 * g + 1] += (uint64_t)r[4 * g + 1] * v.y;
        acc[4 * g + 2] += (uint64_t)r[4 * g + 2] * v.z;
        acc[4 * g + 3] += (uint64_t)r[4 * g + 3] * v.w;
    }
}

// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(RBS) k_ntt_fwd(ModQ m, StageConst sc, const NttTables* __restrict__ tab,
                                                 const int16_t* __restrict__ coef, int64_t npoly,
                                                 uint16_t* __restrict__ out) {
    __shared__ __align__(16) uint32_t xbuf[(RBS / 32) * XWARP];
    const HalfWarp h = half_warp(xbuf);
    LaneTw tw;
    load_lane_tw(tw, tab->w, tab->ws, h.lane);
    for (int64_t base = (int64_t)blockIdx.x * HWB; base < npoly; base += (int64_t)gridDim.x * HWB) {
        const int64_t raw = base + h.slot;
        const bool live = raw < npoly;
        const int64_t item = live ? raw : npoly - 1;
        uint32_t r[EPT];
        int x[EPT];
        load_coef_raw(x, coef + item * D, h.lane);
        ntt_fwd_256_raw(x, r, m, sc, tw, h.xb, h.lane);
#pragma unroll
        for (int i = 0; i < EPT; ++i) r[i] = barrett_full(r[i], m);
        if (live) store_u16x16(out + item * D + 16 * h.lane, r);
    }
}

// The reference's own storage format (parity level L3): Polynomial.ntt_representation is the 2d-point
// CYCLIC transform of the zero-padded coefficient list, natural order, centred: rep[k] = a(zeta^k).
// Odd k = 2i+1 are the negacyclic slots (slot bitrev8(i)); even k = 2m are a(zeta^(2m)), i.e. the
// negacyclic transform of the twisted polynomial c_j * zeta^(-j), slot bitrev8(m).
__global__ void __launch_bounds__(RBS) k_ntt_ref_repr(ModQ m, StageConst sc, const NttTables* __restrict__ tab,
                                                      const int16_t* __restrict__ coef, int64_t npoly,
                                                      int16_t* __restrict__ out) {
    __shared__ __align__(16) uint32_t xbuf[(RBS / 32) * XWARP];
    const HalfWarp h = half_warp(xbuf);
    LaneTw tw;
    load_lane_tw(tw, tab->w, tab->ws, h.lane);
    for (int64_t base = (int64_t)blockIdx.x * HWB; base < npoly; base += (int64_t)gridDim.x * HWB) {
        const int64_t raw = base + h.slot;
        const bool live = raw < npoly;
        const int64_t item = live ? raw : npoly - 1;
        uint32_t odd[EPT], even[EPT];
        load_coef_a(odd, coef + item * D, h.lane, m.cq);
#pragma unroll
        for (int j = 0; j < EPT; ++j) {
            const int idx = h.lane + 16 * j;                          // coefficient index of register j (layout A)
            even[j] = mulmod_full(barrett_full(odd[j], m), tab->pw[(512 - idx) & 511], m) + m.cq;
        }
        ntt_fwd_256(odd, m, sc, tw, h.xb, h.lane);
        ntt_fwd_256(even, m, sc, tw, h.xb, h.lane);
        if (live) {
            int16_t* o = out + item * 2 * D;
#pragma unroll
            for (int k = 0; k < EPT; ++k) {
                const uint32_t i = __brev((uint32_t)(16 * h.lane + k)) >> 24;   // slot p -> exponent index
                o[2 * i + 1] = (int16_t)center(barrett_full(odd[k], m), m);
                o[2 * i] = (int16_t)center(barrett_full(even[k], m), m);
            }
        }
    }
}

__global__ void __launch_bounds__(RBS) k_ntt_inv(ModQ m, StageConst sc, const NttTables* __restrict__ tab,
                                                 const uint16_t* __restrict__ in, int64_t npoly,
                                                 int16_t* __restrict__ coef) {
    __shared__ __align__(16) uint32_t xbuf[(RBS / 32) * XWARP];
    const HalfWarp h = half_warp(xbuf);
    LaneTw itw;
    load_lane_tw(itw, tab->iw, tab->iws, h.lane);
    for (int64_t base = (int64_t)blockIdx.x * HWB; base < npoly; base += (int64_t)gridDim.x * HWB) {
        const int64_t raw = base + h.slot;
        const bool live = raw < npoly;
        const int64_t item = live ? raw : npoly - 1;
        uint32_t r[EPT];
        load_u16x16(r, in + item * D + 16 * h.lane);
        ntt_inv_256(r, m, sc, itw, h.xb, h.lane, m.cq2);
        if (live) store_coef_a(coef + item * D, r, h.lane, m);
    }
}

__global__ void __launch_bounds__(RBS) k_poly_mul(ModQ m, StageConst sc, const NttTables* __restrict__ tab,
                                                  const int16_t* __restrict__ a, const int16_t* __restrict__ b,
                                                  int64_t npoly, int16_t* __restrict__ out) {
    __shared__ __align__(16) uint32_t xbuf[(RBS / 32) * XWARP];
    const HalfWarp h = half_warp(xbuf);
    for (int64_t base = (int64_t)blockIdx.x * HWB; base < npoly; base += (int64_t)gridDim.x * HWB) {
        const int64_t raw = base + h.slot;
        const bool live = raw < npoly;
        const int64_t item = live ? raw : npoly - 1;
        uint32_t ra[EPT], rb[EPT];
        {
            LaneTw tw;
            load_lane_tw(tw, tab->w, tab->ws, h.lane);
            load_coef_a(ra, a + item * D, h.lane, m.cq);
            ntt_fwd_256(ra, m, sc, tw, h.xb, h.lane);
            load_coef_a(rb, b + item * D, h.lane, m.cq);
            ntt_fwd_256(rb, m, sc, tw, h.xb, h.lane);
        }
#pragma unroll
        for (int i = 0; i < EPT; ++i) ra[i] = mulmod_full(barrett_full(ra[i], m), barrett_full(rb[i], m), m);
        LaneTw itw;
        load_lane_tw(itw, tab->iw, tab->iws, h.lane);
        ntt_inv_256(ra, m, sc, itw, h.xb, h.lane, m.cq2);
        if (live) store_coef_a(out + item * D, ra, h.lane, m);
    }
}

// ------------------------------------------------------------------------------------------------
// y = key_ch * v  (v: nvec coefficient-form vectors of l polynomials)
// FP32-assisted per-lane twiddles of stages 5..8 in SHARED memory ({w, wq, cst, kw} per entry, one LDS.128 per
// use): 60 registers fewer than keeping them resident, which buys a fourth resident block per SM.
constexpr int TW_ROW = 15;           // uint4 per lane: 60-word pitch, conflict-free LDS.128
constexpr int TW_BYTES = LANES * TW_ROW * 16;
__device__ __forceinline__ void fill_tw_shared(uint4* twtab, const NttTables* __restrict__ tab) {
    for (int e = threadIdx.x; e < LANES * 15; e += blockDim.x) {
        const int ln = e / 15, i = e % 15;
        const int k = i == 0 ? 16 + ln : (i < 3 ? 32 + 2 * ln + (i - 1) : (i < 7 ? 64 + 4 * ln + (i - 3) : 128 + 8 * ln + (i - 7)));
        twtab[ln * TW_ROW + i] = make_uint4(__ldg(tab->w + k), __float_as_uint(__ldg(tab->f_wq + k)),
                                            __float_as_uint(__ldg(tab->f_cst + k)), __ldg(tab->f_kw + k));
    }
    __syncthreads();
}

__global__ void __launch_bounds__(MBS, 512 / MBS) k_matvec(ModQ m, StageConst sc, StageConstF scf, const NttTables* __restrict__ tab,
                                                const uint32_t* __restrict__ a_hat_g, int l,
                                                const int16_t* __restrict__ vec_coef, int64_t nvec,
                                                uint16_t* __restrict__ vec_ntt, uint16_t* __restrict__ y_ntt,
                                                int16_t* __restrict__ y_coef);

// ------------------------------------------------------------------------------------------------
// Asynchronous global->shared staging (LDGSTS, L2-only) used by k_sign and k_verify: each half-warp owns two
// stage buffers and keeps the next two rows of its work list in flight while it works on the current one, so
// HBM latency never reaches the scoreboard.
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

constexpr int STAGE_HALF_BYTES = 2 * D * 2 + 32;   // two polynomials + 32 B so half-warps differ by 8 banks

// Coefficient-form rows reach k_matvec the way they reach k_verify: through a 2-deep cp.async pipeline per half-warp
// and conflict-free 16-bit shared loads.  (Round 1 read them with 16 strided 2-byte global loads per lane: 35 % of
// the warp samples sat on the long scoreboard.)
__global__ void __launch_bounds__(MBS, 512 / MBS) k_matvec(ModQ m, StageConst sc, StageConstF scf, const NttTables* __restrict__ tab,
                                                const uint32_t* __restrict__ a_hat_g, int l,
                                                const int16_t* __restrict__ vec_coef, int64_t nvec,
                                                uint16_t* __restrict__ vec_ntt, uint16_t* __restrict__ y_ntt,
                                                int16_t* __restrict__ y_coef) {
    extern __shared__ __align__(16) uint32_t smem[];
    uint32_t* a_hat = smem;
    uint32_t* xbuf = smem + l * AROW;
    copy_a_hat(a_hat, a_hat_g, l);
    const HalfWarp h = half_warp(xbuf);
    unsigned char* stage_base = reinterpret_cast<unsigned char*>(xbuf + (MBS / 32) * XWARP);
    unsigned char* stage = stage_base + h.slot * STAGE_HALF_BYTES;
    uint4* twtab = reinterpret_cast<uint4*>(stage_base + MHWB * STAGE_HALF_BYTES);
    fill_tw_shared(twtab, tab);
    const LaneTwFShared twf{twtab + h.lane * TW_ROW};
    const int64_t first = (int64_t)blockIdx.x * MHWB, stride = (int64_t)gridDim.x * MHWB;
    const int64_t trips = first < nvec ? (nvec - first + stride - 1) / stride : 0;   // uniform over the block
    int pf_left = (int)trips;                   // running-pointer prefetch cursor, see k_verify
    int pf_i = 0;
    int64_t pf_item = first + h.slot;
    const unsigned char* const rows_base = reinterpret_cast<const unsigned char*>(vec_coef) + 16 * h.lane;
    const unsigned char* src = rows_base + (pf_item < nvec ? pf_item : nvec - 1) * l * (D * 2);
    const unsigned dst0 = (unsigned)__cvta_generic_to_shared(stage) + 16u * (unsigned)h.lane;
    unsigned pf_off = 0;
    auto issue = [&]() {
        if (pf_left > 0) {
            asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst0 + pf_off), "l"(src) : "memory");
            asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst0 + pf_off + 256), "l"(src + 256) : "memory");
            src += D * 2;
            pf_off ^= (unsigned)(D * 2);
            if (++pf_i == l) {
                pf_i = 0;
                --pf_left;
                pf_item += stride;
                src = pf_item < nvec ? src + (stride - 1) * l * (D * 2) : rows_base + (nvec - 1) * l * (D * 2);
            }
        }
        cp_async_commit();
    };
    issue();
    issue();
    unsigned cur = 0;
    for (int64_t it = 0; it < trips; ++it) {
        const int64_t raw = first + it * stride + h.slot;
        const bool live = raw < nvec;
        const int64_t item = live ? raw : nvec - 1;
        uint64_t acc[EPT];
#pragma unroll
        for (int i = 0; i < EPT; ++i) acc[i] = 0;
        for (int i = 0; i < l; ++i) {
            cp_async_wait<1>();
            __syncwarp();
            uint32_t r[EPT];
            int x[EPT];
            const unsigned sp = (unsigned)__cvta_generic_to_shared(stage + cur * (D * 2) + 2 * h.lane);
#pragma unroll
            for (int j = 0; j < EPT; ++j) asm volatile("ld.shared.s16 %0, [%1];" : "=r"(x[j]) : "r"(sp + 32 * j));
            __syncwarp();
            issue();
            cur ^= 1u;
            ntt_fwd_256_fp(x, r, m, scf, twf, h.xb, h.lane);
#pragma unroll
            for (int k = 0; k < EPT; ++k) r[k] -= FP_BIAS;
            if (vec_ntt) {
#pragma unroll
                for (int k = 0; k < EPT; ++k) r[k] = barrett_full(r[k], m);
                if (live) store_u16x16(vec_ntt + (item * l + i) * D + 16 * h.lane, r);
            }
            mac_row(acc, r, a_hat + i * AROW, h.lane);
        }
        uint32_t y[EPT];
#pragma unroll
        for (int k = 0; k < EPT; ++k) y[k] = reduce64(acc[k], m);
        if (y_ntt && live) store_u16x16(y_ntt + item * D + 16 * h.lane, y);
        if (y_coef) {
            LaneTw itw;
            load_lane_tw(itw, tab->iw, tab->iws, h.lane);
            ntt_inv_256(y, m, sc, itw, h.xb, h.lane, m.cq2);
            if (live) store_coef_a(y_coef + item * D, y, h.lane, m);
        }
    }
}

// k_verify runs 16 warps per SM at 128 registers however they are grouped; grouped as ONE block of 512 threads they share
// one key_ch / twiddle / correction copy (62 instead of 164 KB of shared memory per SM at l = 13; the rest serves the L1
// for the per-item key and challenge loads): 4 x 128 threads 4.075 ms, 2 x 256 3.97 ms, 1 x 512 3.84 ms per 2^20
// (secpar 256, 2^18: 1.73 / 1.68 / 1.64 ms).  Fewer warps lose in proportion - 5 x 96 threads (15 warps) 4.33 ms,
// 7 x 64 (14 warps) 4.65 ms - and more registers or more warps do not pay: 3 x 128 at 155 registers +1.2 %, 5 x 128 at
// 96 registers +1.7 % (profiles/exp_r2_verify_regs.txt).
#ifdef LCB_EXP_VBS
constexpr int VBS = LCB_EXP_VBS;
#else
constexpr int VBS = 512;                 // threads per block of k_verify
#endif
#ifdef LCB_EXP_VERIFY_BLOCKS
constexpr int VERIFY_BLOCKS = LCB_EXP_VERIFY_BLOCKS;
#else
constexpr int VERIFY_BLOCKS = 512 / VBS; // resident blocks per SM k_verify is compiled for (16 warps)
#endif
constexpr int VHWB = VBS / LANES;        // half-warps (items in flight) per block of k_verify

// 16 slots of one lane from a staged 512-byte row.  The row is staged SPLIT: the first 16 bytes of every lane's 32
// (256 bytes), then the second 16 bytes of every lane - so that the eight lanes of a quarter-warp read 128
// contiguous bytes per 128-bit load.  (Staged as it lies in HBM, lane t at byte 32 t, lanes t and t + 4 share their
// banks: a 2-way conflict on every load, 27 % of k_sign's shared wavefronts in round 1.)
__device__ __forceinline__ void load_u16x16_smem(uint32_t (&r)[EPT], const unsigned char* row, int lane) {
    const uint4 a = *reinterpret_cast<const uint4*>(row + 16 * lane);
    const uint4 b = *reinterpret_cast<const uint4*>(row + D + 16 * lane);
    const uint32_t w[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
#pragma unroll
    for (int i = 0; i < 8; ++i) { r[2 * i] = w[i] & 0xFFFFu; r[2 * i + 1] = w[i] >> 16; }
}

constexpr int SIGN_STAGE_BYTES = 2 * (2 * D * 2) + 32;   // two (sk_left row, sk_right row) pairs per half-warp
constexpr int ITW_ROW = 31;           // uint2 {w, w/q} per lane from NttTables::inv_lane: 62-word pitch, conflict-free LDS.64
constexpr int ITW_BYTES = LANES * ITW_ROW * 8;
#ifdef LCB_EXP_SIGN_BLOCKS
constexpr int SIGN_BLOCKS = LCB_EXP_SIGN_BLOCKS;
#else
constexpr int SIGN_BLOCKS = 4;        // resident blocks per SM k_sign is compiled for (121 registers; 5 blocks at 95
                                      // registers: 6.10 instead of 6.03 ms per 2^20, 6 at 80: 6.13 ms)
#endif

// Packed epilogue of k_sign<SIG_BITS>: one row of signature coefficients (lane t holds coefficients t + 16 j after the
// inverse transform) -> 32*SIG_BITS bytes of the wire format (wire.cu) and the row's in_range flag, exactly as k_pack
// would write them from the int16 row.  The half-warp's transposition buffer is free between two transforms and holds
// both stages: (1) the biased 16-bit values in natural order, 16 consecutive values per 12-word group (the pitch makes
// the 128-bit reads of step 2 conflict-free); (2) lane t packs values 16 t .. 16 t + 15 into SIG_BITS halfwords at
// halfword SIG_BITS * t of the packed row; (3) the row leaves in 16-byte coalesced stores (352 / 416 bytes at 11 / 13
// bits are multiples of 16).
constexpr int SIGN_PACK_PITCH = 12;                       // words per group of 16 values
constexpr int SIGN_PACK_ROW = 16 * SIGN_PACK_PITCH;       // word offset of the packed row in the buffer
static_assert(SIGN_PACK_ROW + 8 * 16 <= XHALF, "the packed epilogue must fit the half-warp's transposition buffer");
template <int SIG_BITS>
__device__ __forceinline__ void sign_store_packed(const uint32_t (&a)[EPT], const ModQ& m, uint32_t bias, uint32_t* xb,
                                                  int lane, unsigned mask, bool live, uint8_t* __restrict__ out_row,
                                                  uint8_t* __restrict__ range_flag) {
    uint16_t* v16 = reinterpret_cast<uint16_t*>(xb);
#pragma unroll
    for (int j = 0; j < EPT; ++j) v16[2 * SIGN_PACK_PITCH * j + lane] = (uint16_t)((uint32_t)center_lazy4(a[j], m) + bias);
    __syncwarp();
    const uint4 lo = *reinterpret_cast<const uint4*>(xb + SIGN_PACK_PITCH * lane);
    const uint4 hi = *reinterpret_cast<const uint4*>(xb + SIGN_PACK_PITCH * lane + 4);
    const uint32_t w[8] = {lo.x, lo.y, lo.z, lo.w, hi.x, hi.y, hi.z, hi.w};
    uint16_t* pk = reinterpret_cast<uint16_t*>(xb + SIGN_PACK_ROW) + SIG_BITS * lane;
    constexpr uint32_t LIMIT = 1u << SIG_BITS;
    bool ok = true;
    uint32_t acc = 0;
    int fill = 0, nh = 0;
#pragma unroll
    for (int i = 0; i < 16; ++i) {
        const uint32_t v = (w[i >> 1] >> (16 * (i & 1))) & 0xFFFFu;
        ok = ok && v < LIMIT;
        acc |= (v & (LIMIT - 1)) << fill;
        fill += SIG_BITS;
        if (fill >= 16) {                       // at most one halfword per value: fill < 16 + SIG_BITS <= 32
            pk[nh++] = (uint16_t)acc;
            acc >>= 16;
            fill -= 16;
        }
    }
    __syncwarp();
    if (live) {
        const uint4* src = reinterpret_cast<const uint4*>(xb + SIGN_PACK_ROW);
#pragma unroll
        for (int k = lane; k < 2 * SIG_BITS; k += LANES) reinterpret_cast<uint4*>(out_row)[k] = src[k];
    }
    const unsigned bad = __ballot_sync(0xFFFFFFFFu, !ok) & mask;
    if (live && range_flag && lane == 0) *range_flag = bad ? 0 : 1;
    __syncwarp();                               // the buffer belongs to the next transform again
}

// sig = sk_left ** c + sk_right.  Both transforms are FP32-assisted (round 2): the challenge goes through
// ntt_fwd_256_fp, every row through the decimation-in-time inverse ntt_inv_256_fp, whose closing twist absorbs the
// d^-1 scaling; all per-lane twiddles sit in shared memory.  (Round 1: Shoup butterflies, 96 quarter-rate IMAD.HI per
// row, 7.3 ms per 2^20 with the FMA-heavy pipe as the limiter.)
// SIG_BITS = 0 writes int16 rows to sig; 11 / 13 write packed rows (bias sig_bias) to `sig` read as uint8 and, when
// in_range is not null, one in_range flag per row (sign_store_packed).
template <int SIG_BITS>
__global__ void __launch_bounds__(RBS, SIGN_BLOCKS) k_sign(ModQ m, StageConstF scf, StageConstF iscf, const NttTables* __restrict__ tab, int l,
                                              const uint16_t* __restrict__ sk_ntt, const int16_t* __restrict__ ch_pairs,
                                              int ch_wt, int64_t n, int16_t* __restrict__ sig,
                                              uint8_t* __restrict__ in_range, int sig_bias) {
    extern __shared__ __align__(16) uint32_t smem[];
    uint32_t* xbuf = smem;
    unsigned char* stage = reinterpret_cast<unsigned char*>(xbuf + (RBS / 32) * XWARP);
    uint4* twtab = reinterpret_cast<uint4*>(stage + HWB * SIGN_STAGE_BYTES);
    uint2* itwtab = reinterpret_cast<uint2*>(twtab + LANES * TW_ROW);      // short rows: k_sign is bound by the shared-memory pipeline
    const HalfWarp h = half_warp(xbuf);
    stage += h.slot * SIGN_STAGE_BYTES;
    for (int e = threadIdx.x; e < LANES * ITW_ROW; e += blockDim.x) {
        const uint4 v = __ldg(&tab->inv_lane[0][0] + e);
        itwtab[e] = make_uint2(v.x, v.y);
    }
    fill_tw_shared(twtab, tab);
    const LaneTwFShared twf{twtab + h.lane * TW_ROW};
    const LaneTwFShared2 itwf{itwtab + h.lane * ITW_ROW, m.kw0};
    const int64_t first = (int64_t)blockIdx.x * HWB, stride = (int64_t)gridDim.x * HWB;
    const int64_t trips = first < n ? (n - first + stride - 1) / stride : 0;   // uniform over the block
    // work list of this half-warp: row pair i (sk_left[i], sk_right[i]) of item(it); the cursor runs 2 ahead as a
    // running source pointer (see k_verify)
    int pf_left = (int)trips;
    int pf_i = 0;
    int64_t pf_item = first + h.slot;
    const int64_t item_bytes = (int64_t)2 * l * D * 2, right_off = (int64_t)l * D * 2;
    // The split layout (load_u16x16_smem) puts 16-byte chunk j of a row at (j & 1) * 256 + (j >> 1) * 16.  A lane copies
    // chunks `lane` and `16 + lane`, so that one cp.async instruction reads 256 CONTIGUOUS bytes of the row (the first
    // version had lane t copy its own chunks 2t and 2t + 1: every instruction touched 16 bytes of 16 different sectors and
    // ncu counted 32 shared-memory wavefronts per instruction instead of 7 - half of the kernel's shared traffic).
    const unsigned char* const rows_base = reinterpret_cast<const unsigned char*>(sk_ntt) + 16 * h.lane;
    const unsigned char* src = rows_base + (pf_item < n ? pf_item : n - 1) * item_bytes;
    const unsigned dst0 = (unsigned)__cvta_generic_to_shared(stage) + (unsigned)((h.lane & 1) * D + (h.lane >> 1) * 16);
    unsigned pf_off = 0;
    auto issue = [&]() {
        if (pf_left > 0) {
            const unsigned d = dst0 + pf_off;
            asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(d), "l"(src) : "memory");
            asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(d + 128), "l"(src + D) : "memory");
            asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(d + 2 * D), "l"(src + right_off) : "memory");
            asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(d + 2 * D + 128), "l"(src + right_off + D) : "memory");
            src += D * 2;
            pf_off ^= (unsigned)(2 * D * 2);
            if (++pf_i == l) {
                pf_i = 0;
                --pf_left;
                pf_item += stride;
                src = pf_item < n ? src + stride * item_bytes - right_off : rows_base + (n - 1) * item_bytes;
            }
        }
        cp_async_commit();
    };
    issue();
    issue();
    unsigned cur = 0;
    for (int64_t it = 0; it < trips; ++it) {
        const int64_t raw = first + it * stride + h.slot;
        const bool live = raw < n;
        const int64_t item = live ? raw : n - 1;
        uint32_t c[EPT];
        {
            int cx[EPT];
            load_pairs_raw(cx, ch_pairs + item * ch_wt * 2, ch_wt, h.xb, h.lane);
            ntt_fwd_256_fp(cx, c, m, scf, twf, h.xb, h.lane);
        }
#pragma unroll
        for (int k = 0; k < EPT; ++k) c[k] = barrett_full(c[k] - FP_BIAS, m);
        for (int i = 0; i < l; ++i) {
            cp_async_wait<1>();
            __syncwarp();
            uint32_t a[EPT], b[EPT];
            const unsigned char* rows = stage + cur * (2 * D * 2);
            load_u16x16_smem(a, rows, h.lane);
            load_u16x16_smem(b, rows + D * 2, h.lane);
            __syncwarp();
            issue();                            // refill the buffer just drained with row pair (+2)
            cur ^= 1u;
#pragma unroll
            for (int k = 0; k < EPT; ++k) a[k] = barrett_lazy(c[k] * a[k], m) + b[k] + FP_BIAS;   // < 2q + 2^16, biased
            ntt_inv_256_fp(a, m, iscf, itwf, h.xb, h.lane);
            if constexpr (SIG_BITS == 0) {
                if (live) {
                    int16_t* out = sig + (item * l + i) * D;
#pragma unroll
                    for (int j = 0; j < EPT; ++j) out[h.lane + 16 * j] = (int16_t)center_lazy4(a[j], m);
                }
            } else {
                const int64_t row = item * l + i;
                sign_store_packed<SIG_BITS>(a, m, (uint32_t)sig_bias, h.xb, h.lane, h.mask, live,
                                            reinterpret_cast<uint8_t*>(sig) + row * (32 * SIG_BITS),
                                            in_range ? in_range + row : nullptr);
            }
        }
    }
}

// ------------------------------------------------------------------------------------------------
// verdict = max|v| <= bd && max weight <= wt && key_ch * v == [vk_left * c] + rhs (+ extra)
//   vk_ntt != null : rhs = vk_ntt[item][1], and the challenge term uses vk_ntt[item][0]
//   vk_ntt == null : rhs = rhs_only[item]                               (witness_verify)
// Asynchronous global->shared staging of coefficient-form polynomials (LDGSTS, L2-only): each
// half-warp owns two 512-byte stage buffers and keeps the next two polynomials of its work list
// in flight while it transforms the current one, so HBM latency never reaches the scoreboard.
// 16 NTT slots of one lane from a 14-bit packed polynomial (wire.cu layout): 16 * 14 bits = exactly 7 words
__device__ __forceinline__ void load_u14x16(uint32_t (&r)[EPT], const uint32_t* __restrict__ p) {
    uint32_t w[8];
#pragma unroll
    for (int i = 0; i < 7; ++i) w[i] = __ldg(p + i);
    w[7] = 0;
#pragma unroll
    for (int k = 0; k < EPT; ++k) r[k] = __funnelshift_r(w[(14 * k) >> 5], w[((14 * k) >> 5) + 1], (14 * k) & 31) & 0x3FFFu;
}

// CHECK_WT: weight test, compiled out when wt >= d (every shipped parameter set: vf_wt = d).
// SIG_BITS / VK_BITS: 0 = int16 coefficients / uint16 slots; otherwise the inputs are rows of the packed wire
// format (wire.cu): signatures SIG_BITS bits per coefficient with bias sig_bias, keys VK_BITS (14) bits per slot.
// The packed rows ride through the same cp.async stage buffers and are expanded on the way into registers.
// ST_BITS: 0 = extra_rhs holds uint16 statement slots; 14 = 14-bit packed statements (bias 0, 7 words per lane, read as
// the key halves are).  A 16-bit packed statement has the bytes of a uint16 row and takes ST_BITS = 0.
// RHS_BITS: the same for rhs_only in the witness-verify form (14 = packed adaptor statements).
template <bool CHECK_WT, int SIG_BITS, int VK_BITS, int ST_BITS = 0, int RHS_BITS = 0>
__global__ void __launch_bounds__(VBS, VERIFY_BLOCKS) k_verify(ModQ m, StageConst sc, StageConstF scf, const NttTables* __restrict__ tab,
                                                const uint32_t* __restrict__ a_hat_g, int l,
                                                const int16_t* __restrict__ vec_coef,
                                                const uint16_t* __restrict__ vk_ntt,
                                                const int16_t* __restrict__ ch_pairs, int ch_wt,
                                                const uint16_t* __restrict__ rhs_only,
                                                const uint16_t* __restrict__ extra_rhs, int64_t n, int bd, int wt,
                                                int sig_bias, uint8_t* __restrict__ verdict) {
    constexpr int ROW_BYTES = SIG_BITS ? 32 * SIG_BITS : D * 2;
    extern __shared__ __align__(16) uint32_t smem[];
    uint32_t* a_hat = smem;
    uint32_t* xbuf = smem + l * AROW;
    unsigned char* stage_base = reinterpret_cast<unsigned char*>(xbuf + (VBS / 32) * XWARP);
    copy_a_hat(a_hat, a_hat_g, l);
    const HalfWarp h = half_warp(xbuf);
    unsigned char* stage = stage_base + h.slot * STAGE_HALF_BYTES;
    uint4* twtab = reinterpret_cast<uint4*>(stage_base + VHWB * STAGE_HALF_BYTES);
    fill_tw_shared(twtab, tab);
    const LaneTwFShared twf{twtab + h.lane * TW_ROW};
    // The FP32-assisted transform returns biased values (r + FP_BIAS); the row-vector product then carries
    // FP_BIAS * sum_i a_hat[i][slot], removed once per slot before the comparison.
    // The correction depends on (lane, slot index) only and is used once per item: a 16 x 16 table per block in shared
    // memory (every half-warp writes the same values) instead of 16 registers held across the row loop - the kernel
    // wants 155 registers and is compiled for 128: 4.135 -> 4.06 ms per 2^20 (profiles/exp_r2_verify_regs.txt).
    uint32_t* corr = reinterpret_cast<uint32_t*>(reinterpret_cast<unsigned char*>(twtab) + TW_BYTES) + h.lane;
#define CORR(k) corr[(k) * LANES]
    {
        uint32_t colsum[EPT];
#pragma unroll
        for (int k = 0; k < EPT; ++k) colsum[k] = 0;
        for (int i = 0; i < l; ++i) {
#pragma unroll
            for (int k = 0; k < EPT; ++k) colsum[k] += a_hat[i * AROW + XROW * h.lane + k];
        }
#pragma unroll
        for (int k = 0; k < EPT; ++k) CORR(k) = m.kq18 - mulmod_full(barrett_full(colsum[k], m), m.bias_mod_q, m);
    }
    __syncthreads();            // make the table visible before the first read
    constexpr bool check_wt = CHECK_WT;

    // item indices are 32-bit (the launcher refuses n > 2^30: that many signatures would be terabytes); 64-bit
    // arithmetic only where an address is formed
    const unsigned first = blockIdx.x * VHWB, stride = gridDim.x * VHWB;
    const unsigned n32 = (unsigned)n;
    const int trips = first < n32 ? (int)((n32 - first + stride - 1) / stride) : 0;   // uniform over the block
    // work list of this half-warp: polynomial i of item(it), it = 0..trips-1; the prefetch cursor runs 2 ahead.
    // The cursor is a running source pointer and a running shared-memory address: rows of an item are contiguous, so
    // a row costs one 64-bit add; the item arithmetic (and the clamp of the last, partial trip) runs once per item.
    // (The first version recomputed item, clamp and address for every row: 31 instructions per row, 6.5 % of the kernel.)
    int pf_left = trips;                        // items the cursor has not finished
    int pf_i = 0;
    unsigned pf_item = first + h.slot;
    const unsigned char* const rows_base = reinterpret_cast<const unsigned char*>(vec_coef) + 16 * h.lane;
    const unsigned char* src = rows_base + (int64_t)(pf_item < n32 ? pf_item : n32 - 1) * l * ROW_BYTES;
    const unsigned dst0 = (unsigned)__cvta_generic_to_shared(stage) + 16u * (unsigned)h.lane;
    unsigned pf_off = 0;
    auto issue = [&]() {
        if (pf_left > 0) {
            LCB_CHECK(src >= rows_base && (src - rows_base) + ROW_BYTES <= n * l * ROW_BYTES);   // a row of the batch
#pragma unroll
            for (int o = 0; o < ROW_BYTES; o += 16 * LANES)
                if (o + 16 * h.lane < ROW_BYTES)
                    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst0 + pf_off + o), "l"(src + o) : "memory");
            src += ROW_BYTES;
            pf_off ^= (unsigned)(D * 2);
            if (++pf_i == l) {
                pf_i = 0;
                --pf_left;
                pf_item += stride;
                src = pf_item < n32 ? src + (int64_t)(stride - 1) * l * ROW_BYTES : rows_base + (int64_t)(n32 - 1) * l * ROW_BYTES;
            }
        }
        cp_async_commit();
    };
    issue();
    issue();
    unsigned cur = 0;
    unsigned raw = first + h.slot;
    for (int it = 0; it < trips; ++it, raw += stride) {
        const bool live = raw < n32;
        const int64_t item = live ? raw : n32 - 1;
        uint64_t acc[EPT];
#pragma unroll
        for (int i = 0; i < EPT; ++i) acc[i] = 0;
        bool bad = false;
        int hi = 0, lo = 0;                     // running max / min coefficient of the whole vector
        for (int i = 0; i < l; ++i) {
            cp_async_wait<1>();
            __syncwarp();
            int pre[EPT];
            if (SIG_BITS == 0) {
                const unsigned sp = (unsigned)__cvta_generic_to_shared(stage + cur * (D * 2) + 2 * h.lane);
#pragma unroll
                for (int j = 0; j < EPT; ++j)      // sign-extending 16-bit shared load (plain C++ yields LDS.U16 + PRMT)
                    asm volatile("ld.shared.s16 %0, [%1];" : "=r"(pre[j]) : "r"(sp + 32 * j));
            } else {
                // coefficient lane + 16 j sits at bit (lane + 16 j) * SIG_BITS of the row: the word offset of j is a
                // compile-time constant on top of one of two per-lane (word, shift) pairs (16 * SIG_BITS is a
                // multiple of 16 bits, so the in-word phase alternates between two values)
                const unsigned row = (unsigned)__cvta_generic_to_shared(stage + cur * (D * 2));
                const unsigned b0 = (unsigned)h.lane * SIG_BITS, b1 = b0 + 16;
                const unsigned sp0 = row + 4 * (b0 >> 5), sp1 = row + 4 * (b1 >> 5), sh0 = b0 & 31, sh1 = b1 & 31;
#pragma unroll
                for (int j = 0; j < EPT; ++j) {
                    const int c = 16 * SIG_BITS * j;              // bit offset of j relative to j = 0
                    const bool odd = (c & 31) != 0;               // then c = 32 k + 16
                    const unsigned a = (odd ? sp1 : sp0) + 4 * (unsigned)((c - (odd ? 16 : 0)) >> 5);
                    uint32_t lo_w, hi_w;
                    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(lo_w) : "r"(a));
                    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(hi_w) : "r"(a + 4));
                    pre[j] = (int)(__funnelshift_r(lo_w, hi_w, odd ? sh1 : sh0) & ((1u << SIG_BITS) - 1)) - sig_bias;
                }
            }
            __syncwarp();
            issue();                            // refill the buffer just drained with polynomial (+2)
            cur ^= 1u;
            uint32_t r[EPT];
#pragma unroll
            for (int j = 0; j < EPT; j += 2) {
                hi = __vimax3_s32(hi, pre[j], pre[j + 1]);
                lo = __vimin3_s32(lo, pre[j], pre[j + 1]);
            }
            if (check_wt) {
                int nz = 0;
#pragma unroll
                for (int j = 0; j < EPT; ++j) nz += (pre[j] != 0);
#pragma unroll
                for (int o = 8; o >= 1; o >>= 1) nz += __shfl_xor_sync(0xFFFFFFFFu, nz, o);
                bad |= nz > wt;
            }
            ntt_fwd_256_fp(pre, r, m, scf, twf, h.xb, h.lane);
            mac_row(acc, r, a_hat + i * AROW, h.lane);
        }
        bad |= hi > bd || lo < -bd;
        uint32_t rhs[EPT];
        if (vk_ntt) {
            uint32_t c[EPT], vl[EPT];
            int cx[EPT];
            load_pairs_raw(cx, ch_pairs + item * ch_wt * 2, ch_wt, h.xb, h.lane);
            ntt_fwd_256_fp(cx, c, m, scf, twf, h.xb, h.lane);
            if (VK_BITS == 14) {
                const uint32_t* vp = reinterpret_cast<const uint32_t*>(vk_ntt) + item * (2 * 112) + 7 * h.lane;
                load_u14x16(vl, vp);
                load_u14x16(rhs, vp + 112);
            } else {
                load_u16x16(vl, vk_ntt + item * 2 * D + 16 * h.lane);
                load_u16x16(rhs, vk_ntt + item * 2 * D + D + 16 * h.lane);
            }
#pragma unroll
            for (int k = 0; k < EPT; ++k) acc[k] += (uint64_t)(c[k] - FP_BIAS) * (m.cq2 - vl[k]);
        } else if (RHS_BITS == 14) {
            load_u14x16(rhs, reinterpret_cast<const uint32_t*>(rhs_only) + item * 112 + 7 * h.lane);
        } else {
            load_u16x16(rhs, rhs_only + item * D + 16 * h.lane);
        }
        if (extra_rhs) {
            uint32_t ex[EPT];
            if (ST_BITS == 14)
                load_u14x16(ex, reinterpret_cast<const uint32_t*>(extra_rhs) + item * 112 + 7 * h.lane);
            else
                load_u16x16(ex, extra_rhs + item * D + 16 * h.lane);
#pragma unroll
            for (int k = 0; k < EPT; ++k) rhs[k] += ex[k];
        }
        bool eq = true;
#pragma unroll
        for (int k = 0; k < EPT; ++k) eq &= divisible_by_q(acc[k] + (uint64_t)(CORR(k) - rhs[k]), m);   // corr = kq18 - bias term
        const unsigned votes = __ballot_sync(0xFFFFFFFFu, eq && !bad);
        if (live && h.lane == 0) verdict[item] = (votes & h.mask) == h.mask ? 1 : 0;
    }
}

// ------------------------------------------------------------------------------------------------
// k_verify_tc: the same verdict for int16 rows, with key_ch * v as two exact u8 tensor-core GEMMs (DESIGN.md section 3.3).
// With zeta = psi^128, slot p < 128 of NTT(a) evaluates u0 = a_lo + zeta a_hi and slot p >= 128 evaluates
// u1 = a_lo - zeta a_hi (a_lo / a_hi: coefficients 0..127 / 128..255) at 128 points, so for block b
//   sum_k key_hat_k[p] s_hat_k[p] = sum_(k, m) M_b[p][(k, m)] u^b_k[m],   M_b[p][(k, m)] = key_hat_k[p] x_p^m mod q.
// The CUDA cores form u < 2^16 congruent to it mod q (tc_limbs_reduce) and split it into two u8 limbs (A = [u & 255 |
// u >> 8], K = 2 * 128 * l); the context holds B_b = [M_b ; 256 M_b mod q] split into byte columns (N = 2 * 128:
// slot x (lo, hi)), built by k_verify_tc_matrix.
// D_b = A B_b^T then gives x[p] = D_lo[p] + 256 D_hi[p] = sum_k key_hat_k[p] s_hat_k[p] (mod q), exactly: every entry is
// below 255 * 255 * 256 * l < 2^31 for l <= 128 (contexts take l <= 64).
//
// One CTA per SM, 128 verifies (= the 128 tensor-memory lanes) per tile, both blocks accumulated at once in all 512
// columns.  K runs in chunks of 64 bytes per block - (poly k, quarter mq: m in 32 mq .. 32 mq + 31) x (limb 0, limb 1) -
// through TC_STAGES shared-memory stages.  Roles:
//   warps 0-3   right-hand sides of the tile (half-warp NTT of the challenge, as k_verify), then the epilogue: thread r
//               reads tensor-memory lane r (its verify) and tests x - rhs for divisibility by q at every slot;
//   warp 4      bulk copies of the B chunks (L2-resident, read by every CTA);
//   warp 5      tensor-memory allocation and the MMA-issuing thread;
//   warps 6-13  converters: thread (r, h) reads 16 coefficient pairs of verify r per stage from HBM, keeps the running
//               bound / weight checks, and writes the u limbs of both blocks into the A stage.
constexpr int TC_ROWS = 128;
constexpr int TC_STAGES = 3;
constexpr int TC_A_BLOCK = TC_ROWS * 64;                  // bytes of one block's A chunk (128 rows x 64 K-bytes)
constexpr int TC_B_BLOCK = 256 * 64;                      // bytes of one block's B chunk (256 columns x 64 K-bytes)
constexpr int TC_B_CHUNK = 2 * TC_B_BLOCK;                // bytes of B per K chunk (both blocks), one bulk copy
constexpr int TC_STAGE_BYTES = 2 * TC_A_BLOCK + TC_B_CHUNK;
constexpr int TC_RHS_PITCH = D / 2 + 1;                   // words per rhs row: the epilogue's 32 rows fall in 32 banks
constexpr int TC_EPI_WARPS = 4, TC_CONV_WARPS = 8;
constexpr int TC_MIN_TILES_PER_SM = 1;                   // batches below one tile per SM stay on k_verify
constexpr int TC_THREADS = 32 * (TC_EPI_WARPS + 2 + TC_CONV_WARPS);
constexpr size_t tc_smem_bytes() {
    return (size_t)TC_STAGES * TC_STAGE_BYTES + (size_t)TC_ROWS * TC_RHS_PITCH * 4 + (size_t)TW_BYTES +
           (size_t)TC_EPI_WARPS * XWARP * 4 + 2 * TC_ROWS + 8 * (2 * TC_STAGES + 2) + 16;
}

// B_b in the stage layout: K chunk g = 4 k + mq holds [block 0 | block 1], each 4 K-columns of 16 bytes x 256 rows n =
// 128 hl + p; byte kb = 32 L + (m - 32 mq) of row n is byte hl of 256^L key_hat_k[P] x_P^m mod q, P = 128 b + p.
__global__ void k_verify_tc_matrix(ModQ m, const NttTables* __restrict__ tab, const uint32_t* __restrict__ a_hat, int l,
                                   uint8_t* __restrict__ out) {
    const int64_t total = (int64_t)l * 4 * TC_B_CHUNK;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int g = (int)(i / TC_B_CHUNK), rem = (int)(i % TC_B_CHUNK);
        const int b = rem / TC_B_BLOCK, off = rem % TC_B_BLOCK;
        const int kb = (off >> 12) * 16 + (off & 15), n = (off >> 4) & 255;
        const int L = kb >> 5, mm = 32 * (g & 3) + (kb & 31), k = g >> 2;
        const int P = 128 * b + (n & 127);
        uint64_t v = (uint64_t)a_hat[k * D + P] * tab->pw[((uint32_t)tab->oddexp[P] * (uint32_t)mm) & 511] % m.q;
        if (L) v = v * 256 % m.q;
        out[i] = (uint8_t)((n >> 7) ? v >> 8 : v & 255);
    }
}

// u only has to be congruent to a_lo +- zeta a_hi mod q and below 2^16 (two u8 limbs): D_lo + 256 D_hi is then congruent
// to the key_ch product, which is all the epilogue tests, and every D entry keeps its bound.  barrett_lazy lands in
// [0, 2q), so for q <= 32768 (LAZY) it is reduced enough; larger q take one conditional subtraction.
template <bool LAZY>
__device__ __forceinline__ uint32_t tc_limbs_reduce(uint32_t x, const ModQ& m) {
    return LAZY ? barrett_lazy(x, m) : csub(barrett_lazy(x, m), m.q);
}

template <bool CHECK_WT, bool LAZY>
__global__ void __launch_bounds__(TC_THREADS, 1) k_verify_tc(ModQ m, StageConstF scf, const NttTables* __restrict__ tab,
                                                   const uint8_t* __restrict__ bmat, int l,
                                                   const int16_t* __restrict__ vec_coef, const uint16_t* __restrict__ vk_ntt,
                                                   const int16_t* __restrict__ ch_pairs, int ch_wt,
                                                   const uint16_t* __restrict__ rhs_only,
                                                   const uint16_t* __restrict__ extra_rhs, int64_t n, int bd, int wt,
                                                   uint32_t zeta, uint32_t kz0, uint32_t kz1, uint8_t* __restrict__ verdict) {
    extern __shared__ __align__(128) unsigned char tc_smem[];
    unsigned char* stages = tc_smem;
    uint32_t* rhs_buf = reinterpret_cast<uint32_t*>(stages + TC_STAGES * TC_STAGE_BYTES);
    uint4* twtab = reinterpret_cast<uint4*>(rhs_buf + TC_ROWS * TC_RHS_PITCH);
    uint32_t* xbuf = reinterpret_cast<uint32_t*>(reinterpret_cast<unsigned char*>(twtab) + TW_BYTES);
    uint8_t* badbuf = reinterpret_cast<uint8_t*>(xbuf + TC_EPI_WARPS * XWARP);     // [2][128], by tile parity
    uint64_t* full = reinterpret_cast<uint64_t*>(badbuf + 2 * TC_ROWS);
    uint64_t* empty = full + TC_STAGES;
    uint64_t* acc_full = empty + TC_STAGES;
    uint64_t* acc_empty = acc_full + 1;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_empty + 1);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (threadIdx.x == 0) {
        for (int s = 0; s < TC_STAGES; ++s) {
            mbar_init(&full[s], TC_CONV_WARPS + 1);     // converter warps + the B copy (arrive.expect_tx)
            mbar_init(&empty[s], 1);                    // MMA commit
        }
        mbar_init(acc_full, 2);                         // MMA commit + the MMA thread (orders the bound flags)
        mbar_init(acc_empty, TC_EPI_WARPS * 32);
        mbar_init_fence();
    }
    if (warp == TC_EPI_WARPS + 1) {
        tmem_alloc(tmem_slot, 512);
        tc_fence_before();
    }
    fill_tw_shared(twtab, tab);                         // ends in __syncthreads
    tc_fence_after();
    const uint32_t tmem = *tmem_slot;

    const uint32_t n32 = (uint32_t)n;
    const uint32_t tiles = (n32 + TC_ROWS - 1) / TC_ROWS;
    const int chunks = 4 * l;                           // K chunks per tile

    if (warp < TC_EPI_WARPS) {
        // ---- right-hand sides, then the epilogue
        const HalfWarp h = half_warp(xbuf);
        const LaneTwFShared twf{twtab + h.lane * TW_ROW};
        const int r = threadIdx.x;
        int t = 0;
        for (uint32_t tile = blockIdx.x; tile < tiles; tile += gridDim.x, ++t) {
            asm volatile("bar.sync 1, %0;" ::"n"(TC_EPI_WARPS * 32) : "memory");    // rhs_buf of the last tile is read
            for (int row = h.slot; row < TC_ROWS; row += 2 * TC_EPI_WARPS) {
                const uint32_t raw = tile * TC_ROWS + row;
                const int64_t item = raw < n32 ? raw : n32 - 1;
                uint32_t rhs[EPT];
                if (vk_ntt) {
                    uint32_t c[EPT], vl[EPT];
                    int cx[EPT];
                    load_pairs_raw(cx, ch_pairs + item * ch_wt * 2, ch_wt, h.xb, h.lane);
                    ntt_fwd_256_fp(cx, c, m, scf, twf, h.xb, h.lane);
                    load_u16x16(vl, vk_ntt + item * 2 * D + 16 * h.lane);
                    load_u16x16(rhs, vk_ntt + item * 2 * D + D + 16 * h.lane);
#pragma unroll
                    for (int k = 0; k < EPT; ++k) rhs[k] += mulmod_full(barrett_full(c[k] - FP_BIAS, m), vl[k], m);
                } else {
                    load_u16x16(rhs, rhs_only + item * D + 16 * h.lane);
                }
                if (extra_rhs) {
                    uint32_t ex[EPT];
                    load_u16x16(ex, extra_rhs + item * D + 16 * h.lane);
#pragma unroll
                    for (int k = 0; k < EPT; ++k) rhs[k] += ex[k];
                }
                uint32_t* dst = rhs_buf + row * TC_RHS_PITCH + 8 * h.lane;
#pragma unroll
                for (int k = 0; k < EPT; k += 2) dst[k / 2] = barrett_full(rhs[k], m) | (barrett_full(rhs[k + 1], m) << 16);
            }
            asm volatile("bar.sync 1, %0;" ::"n"(TC_EPI_WARPS * 32) : "memory");    // every rhs row of this tile written
            mbar_wait(acc_full, t & 1);
            tc_fence_after();
            bool eq = true;
            const uint32_t* my = rhs_buf + r * TC_RHS_PITCH;
            const uint32_t lane_base = tmem + ((uint32_t)(32 * warp) << 16);
#pragma unroll 1
            for (int col = 0; col < 2 * 128; col += 16) {           // col = 128 b + p0
                const int b = col >> 7, p0 = col & 127;
                uint32_t lo[16], hi[16];
                tmem_ld16(lane_base + 256 * b + p0, lo);
                tmem_ld16(lane_base + 256 * b + 128 + p0, hi);
                tmem_ld_wait();
#pragma unroll
                for (int j = 0; j < 16; j += 2) {
                    const uint32_t w = my[(col + j) >> 1];
                    eq &= divisible_by_q((uint64_t)lo[j] + ((uint64_t)hi[j] << 8) + (m.q - (w & 0xFFFFu)), m);
                    eq &= divisible_by_q((uint64_t)lo[j + 1] + ((uint64_t)hi[j + 1] << 8) + (m.q - (w >> 16)), m);
                }
            }
            tc_fence_before();
            mbar_arrive(acc_empty);
            const uint32_t raw = tile * TC_ROWS + r;
            if (raw < n32) verdict[raw] = (eq && !badbuf[(t & 1) * TC_ROWS + r]) ? 1 : 0;
        }
    } else if (warp == TC_EPI_WARPS) {
        // ---- B chunks
        if (lane == 0) {
            uint32_t s = 0;
            for (uint32_t tile = blockIdx.x; tile < tiles; tile += gridDim.x)
                for (int g = 0; g < chunks; ++g, ++s) {
                    const uint32_t slot = s % TC_STAGES, round = s / TC_STAGES;
                    if (round > 0) mbar_wait(&empty[slot], (round - 1) & 1);
                    mbar_arrive_tx(&full[slot], TC_B_CHUNK);
                    bulk_g2s(stages + slot * TC_STAGE_BYTES + 2 * TC_A_BLOCK, bmat + (size_t)g * TC_B_CHUNK, TC_B_CHUNK,
                             &full[slot]);
                }
        }
    } else if (warp == TC_EPI_WARPS + 1) {
        // ---- MMA issue
        if (lane == 0) {
            constexpr uint32_t idesc = umma_idesc_u8(TC_ROWS, 256);
            uint32_t s = 0;
            int t = 0;
            for (uint32_t tile = blockIdx.x; tile < tiles; tile += gridDim.x, ++t) {
                if (t > 0) {
                    mbar_wait(acc_empty, (t - 1) & 1);
                    tc_fence_after();
                }
                for (int g = 0; g < chunks; ++g, ++s) {
                    const uint32_t slot = s % TC_STAGES, round = s / TC_STAGES;
                    mbar_wait(&full[slot], round & 1);
                    tc_fence_after();
                    const uint32_t a0 = smem_addr(stages + slot * TC_STAGE_BYTES), b0 = a0 + 2 * TC_A_BLOCK;
#pragma unroll
                    for (int b = 0; b < 2; ++b)
#pragma unroll
                        for (int L = 0; L < 2; ++L)
                            umma_u8(tmem + 256 * b, umma_desc(a0 + b * TC_A_BLOCK + L * 2 * (16 * TC_ROWS), 16 * TC_ROWS, 128),
                                    umma_desc(b0 + b * TC_B_BLOCK + L * 2 * (16 * 256), 16 * 256, 128), idesc, g > 0 || L > 0);
                    umma_commit(&empty[slot]);
                }
                umma_commit(acc_full);
                mbar_arrive(acc_full);
            }
        }
    } else {
        // ---- converters: thread (r, hh) owns coefficient pairs m in 32 mq + 16 hh + [0, 16) of verify r in every chunk
        const int ct = threadIdx.x - 32 * (TC_EPI_WARPS + 2);
        const int r = ct >> 1, hh = ct & 1;
        const uint32_t zn = m.q - zeta;
        const int lim_hi = 32768 + bd, lim_lo = 32768 - bd;     // on the biased values a + 32768
        uint32_t s = 0;
        int t = 0;
        // one chunk ahead in registers: 16 low and 16 high coefficients
        uint4 nx[4];
        auto load = [&](uint32_t tile, int g) {
            const uint32_t raw = tile * TC_ROWS + r;
            const int64_t item = raw < n32 ? raw : n32 - 1;
            const int16_t* row = vec_coef + (item * l + (g >> 2)) * D + 32 * (g & 3) + 16 * hh;
            LCB_CHECK(row >= vec_coef && row + D / 2 + 16 <= vec_coef + n * l * D);
            const uint4* p = reinterpret_cast<const uint4*>(row);
            const uint4* q = reinterpret_cast<const uint4*>(row + D / 2);
            nx[0] = __ldg(p);
            nx[1] = __ldg(p + 1);
            nx[2] = __ldg(q);
            nx[3] = __ldg(q + 1);
        };
        if (blockIdx.x < tiles) load(blockIdx.x, 0);
        for (uint32_t tile = blockIdx.x; tile < tiles; tile += gridDim.x, ++t) {
            uint32_t mx = 0, mn = 0xFFFFFFFFu;                  // running max / min of the biased halves
            bool heavy = false;
            int nz = 0;
            for (int g = 0; g < chunks; ++g, ++s) {
                const uint4 cur[4] = {nx[0], nx[1], nx[2], nx[3]};
                if (g + 1 < chunks) load(tile, g + 1);
                else if (tile + gridDim.x < tiles) load(tile + gridDim.x, 0);
                const uint32_t wl[8] = {cur[0].x, cur[0].y, cur[0].z, cur[0].w, cur[1].x, cur[1].y, cur[1].z, cur[1].w};
                const uint32_t wh[8] = {cur[2].x, cur[2].y, cur[2].z, cur[2].w, cur[3].x, cur[3].y, cur[3].z, cur[3].w};
                uint32_t o[2][2][4];                            // [block][limb][word]
#pragma unroll
                for (int w4 = 0; w4 < 4; ++w4) {
                    uint32_t u[2][4];
#pragma unroll
                    for (int w = 0; w < 2; ++w) {
                        const uint32_t bl = wl[2 * w4 + w] ^ 0x80008000u, bh = wh[2 * w4 + w] ^ 0x80008000u;
                        mx = __vmaxu2(mx, __vmaxu2(bl, bh));
                        mn = __vminu2(mn, __vminu2(bl, bh));
                        if (CHECK_WT)
                            nz += ((bl & 0xFFFFu) != 0x8000u) + ((bl >> 16) != 0x8000u) + ((bh & 0xFFFFu) != 0x8000u) +
                                  ((bh >> 16) != 0x8000u);
#pragma unroll
                        for (int e = 0; e < 2; ++e) {
                            const uint32_t lo = e ? bl >> 16 : bl & 0xFFFFu, hi = e ? bh >> 16 : bh & 0xFFFFu;
                            u[0][2 * w + e] = tc_limbs_reduce<LAZY>(hi * zeta + (lo + kz0), m);
                            u[1][2 * w + e] = tc_limbs_reduce<LAZY>(hi * zn + (lo + kz1), m);
                        }
                    }
#pragma unroll
                    for (int b = 0; b < 2; ++b) {
                        const uint32_t p01 = __byte_perm(u[b][0], u[b][1], 0x5410), p23 = __byte_perm(u[b][2], u[b][3], 0x5410);
                        o[b][0][w4] = __byte_perm(p01, p23, 0x6420);
                        o[b][1][w4] = __byte_perm(p01, p23, 0x7531);
                    }
                }
                if (CHECK_WT && (g & 3) == 3) {                 // the row (poly g / 4) is complete over the pair
                    heavy |= nz + __shfl_xor_sync(0xFFFFFFFFu, nz, 1) > wt;
                    nz = 0;
                }
                const uint32_t slot = s % TC_STAGES, round = s / TC_STAGES;
                if (g + 1 == chunks) {                          // bound flags of the tile, before its last chunk is signalled
                    const uint32_t MX = max(mx & 0xFFFFu, mx >> 16), MN = min(mn & 0xFFFFu, mn >> 16);
                    bool bad = heavy || (int)MX > lim_hi || (int)MN < lim_lo;
                    bad |= __shfl_xor_sync(0xFFFFFFFFu, (int)bad, 1) != 0;
                    if (hh == 0) badbuf[(t & 1) * TC_ROWS + r] = bad ? 1 : 0;
                }
                if (round > 0) mbar_wait(&empty[slot], (round - 1) & 1);
                unsigned char* a = stages + slot * TC_STAGE_BYTES + 16 * r;
#pragma unroll
                for (int b = 0; b < 2; ++b)
#pragma unroll
                    for (int L = 0; L < 2; ++L)
                        *reinterpret_cast<uint4*>(a + b * TC_A_BLOCK + (2 * L + hh) * (16 * TC_ROWS)) =
                            make_uint4(o[b][L][0], o[b][L][1], o[b][L][2], o[b][L][3]);
                fence_async_smem();
                __syncwarp();
                if (lane == 0) mbar_arrive(&full[slot]);
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == TC_EPI_WARPS + 1) {
        tc_fence_after();
        tmem_free(tmem, 512);
    }
}

// ------------------------------------------------------------------------------------------------
__global__ void k_vec_addsub(ModQ m, const int16_t* __restrict__ a, const int16_t* __restrict__ b, int64_t nelem,
                             int sub, int16_t* __restrict__ out) {
    // 8 coefficients (16 bytes) per thread per step
    const int64_t nvec = nelem / 8;
    const uint4* a4 = reinterpret_cast<const uint4*>(a);
    const uint4* b4 = reinterpret_cast<const uint4*>(b);
    uint4* o4 = reinterpret_cast<uint4*>(out);
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nvec; i += (int64_t)gridDim.x * blockDim.x) {
        uint4 va = __ldg(a4 + i), vb = __ldg(b4 + i), vo;
        const uint32_t wa[4] = {va.x, va.y, va.z, va.w}, wb[4] = {vb.x, vb.y, vb.z, vb.w};
        uint32_t wo[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            int a0 = (int16_t)(wa[k] & 0xFFFF), a1 = (int16_t)(wa[k] >> 16);
            int b0 = (int16_t)(wb[k] & 0xFFFF), b1 = (int16_t)(wb[k] >> 16);
            if (sub) { b0 = -b0; b1 = -b1; }
            int r0 = center(barrett_full((uint32_t)(a0 + b0 + 2 * (int)m.cq + (int)m.q), m), m);
            int r1 = center(barrett_full((uint32_t)(a1 + b1 + 2 * (int)m.cq + (int)m.q), m), m);
            wo[k] = ((uint32_t)r0 & 0xFFFFu) | ((uint32_t)r1 << 16);
        }
        vo = make_uint4(wo[0], wo[1], wo[2], wo[3]);
        o4[i] = vo;
    }
}

// ------------------------------------------------------------------------------------------------
// BKLM aggregate, monomial coefficients: partial[i][p] += s * sig[t][i][(p - k) mod 256] * (p < k ? -1 : 1)
// A pure HBM stream (512 bytes per polynomial, one add per 2 bytes) - provided the rotation costs next to nothing.
// grid = (chunks, l); a warp keeps AGG_DEPTH rows of its polynomial in flight (one coalesced 16-byte load per lane and
// row).  A row is parked in shared memory TWICE, as E = [~row | row] (512 int16): output position p of a row rotated by
// k then sits at E[256 + p - k] whatever p and k are - no wrap-around, no comparison, no select: per row and lane 8
// sign-extending 16-bit shared loads at immediate offsets (consecutive lanes read consecutive halfwords: conflict-free)
// and 8 multiply-adds.  The wrapped positions read ~v = -v - 1 instead of -v; the missing "+ s" per wrapped read depends
// only on (k, s) of the row, not on the data: hist[k] += s once per row, and at the end of the block
// corr[p] = sum over k > p of hist[k] is added to every position.  (Round 1 read the rotated positions from global
// memory 2 bytes at a time: 2.36 TB/s; the first shared-memory version spent 103 instructions per row on index
// wrap-around, compare and select and was issue-bound at 3.55 TB/s.)
constexpr int AGG_WARPS = 8;
constexpr int AGG_DEPTH = 4;
__global__ void __launch_bounds__(32 * AGG_WARPS, 4) k_agg_partial(ModQ m, int l, const int16_t* __restrict__ sigs,
                                                               const int16_t* __restrict__ ag_pairs, int64_t count,
                                                               int32_t* __restrict__ partial) {
    __shared__ int32_t red[D];
    __shared__ int32_t hist[D];
    __shared__ int32_t wsum[AGG_WARPS];
    __shared__ __align__(16) int16_t rows[AGG_WARPS][AGG_DEPTH][2 * D];
    const int poly = blockIdx.y;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    red[threadIdx.x] = 0;
    hist[threadIdx.x] = 0;
    __syncthreads();
    int32_t acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    const uint32_t* ap = reinterpret_cast<const uint32_t*>(ag_pairs);
    const int64_t stride = (int64_t)gridDim.x * AGG_WARPS;
    uint4 v[AGG_DEPTH];
    uint32_t pr[AGG_DEPTH];
    // rows of this warp: t0, t0 + stride, ...; `left` of them remain (32-bit: count / stride fits easily)
    const int64_t t0 = (int64_t)blockIdx.x * AGG_WARPS + warp;
    int left = t0 < count ? (int)((count - t0 + stride - 1) / stride) : 0;
    const unsigned char* rowp = reinterpret_cast<const unsigned char*>(sigs + (t0 * l + poly) * D) + 16 * lane;
    const uint32_t* app = ap + t0;
    const int64_t rstep = stride * l * (D * 2);
    auto fetch = [&]() {                         // the next min(left, AGG_DEPTH) rows; missing rows read as (0, sign 0)
        if (left >= AGG_DEPTH) {
#pragma unroll
            for (int j = 0; j < AGG_DEPTH; ++j) {
                v[j] = __ldg(reinterpret_cast<const uint4*>(rowp + j * rstep));
                pr[j] = __ldg(app + j * stride);
            }
        } else {
#pragma unroll
            for (int j = 0; j < AGG_DEPTH; ++j) {
                v[j] = make_uint4(0, 0, 0, 0);
                pr[j] = 0;
                if (j < left) {
                    v[j] = __ldg(reinterpret_cast<const uint4*>(rowp + j * rstep));
                    pr[j] = __ldg(app + j * stride);
                }
            }
        }
        LCB_CHECK(left <= 0 || (t0 + (int64_t)(left - 1) * stride < count && poly < l));
        rowp += AGG_DEPTH * rstep;
        app += AGG_DEPTH * stride;
    };
    if (left > 0) fetch();
    const unsigned rows_s = (unsigned)__cvta_generic_to_shared(rows[warp][0]);
    while (left > 0) {
        uint32_t cur[AGG_DEPTH];
#pragma unroll
        for (int j = 0; j < AGG_DEPTH; ++j) {
            uint4* e = reinterpret_cast<uint4*>(rows[warp][j]);
            e[lane] = make_uint4(~v[j].x, ~v[j].y, ~v[j].z, ~v[j].w);
            e[32 + lane] = v[j];
            cur[j] = pr[j];
        }
        __syncwarp();
        left -= AGG_DEPTH;
        if (left > 0) fetch();                   // next rows in flight while this batch is folded
#pragma unroll
        for (int j = 0; j < AGG_DEPTH; ++j) {
            const int k = (int)(cur[j] & 0xFF);
            const int sg = (int)(int16_t)(cur[j] >> 16);
            const unsigned a = rows_s + (unsigned)(j * 4 * D) + 2u * (unsigned)(D - k + lane);
#pragma unroll
            for (int jj = 0; jj < 8; ++jj) {
                int x;
                asm volatile("ld.shared.s16 %0, [%1];" : "=r"(x) : "r"(a + 64u * jj));
                acc[jj] += sg * x;
            }
            if (lane == 0 && sg != 0) atomicAdd(&hist[k], sg);
        }
        __syncwarp();
    }
#pragma unroll
    for (int jj = 0; jj < 8; ++jj) atomicAdd(&red[lane + 32 * jj], acc[jj]);
    __syncthreads();
    {
        // corr[p] = sum_{k > p} hist[k]: suffix sums inside the warp, then the totals of the warps above
        const int p = threadIdx.x;
        const int own = hist[p];
        int sfx = own;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int y = __shfl_down_sync(0xFFFFFFFFu, sfx, o);
            if (lane + o < 32) sfx += y;
        }
        if (lane == 0) wsum[warp] = sfx;
        __syncthreads();
        int above = 0;
        for (int w = warp + 1; w < AGG_WARPS; ++w) above += wsum[w];
        int v = (red[p] + sfx - own + above) % (int)m.q;   // keep cross-block / cross-rank sums far from int32 overflow
        atomicAdd(&partial[poly * D + p], v);
    }
}

__global__ void k_agg_finish(ModQ m, const int32_t* __restrict__ partial, int n, int16_t* __restrict__ out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    int v = partial[i] % (int)m.q;
    if (v < 0) v += (int)m.q;
    out[i] = (int16_t)center((uint32_t)v, m);
}

// BKLM aggregate_verify right-hand side: partial[p] += (vk_left*c + vk_right)[p] * (s * X^k)^(p), NTT form.
// Round 2: the challenge goes through the FP32-assisted transform (no quarter-rate IMAD.HI in the butterflies), the
// monomial's sign is folded into the exponent (psi^256 = -1: -psi^e = psi^(e+256)), products are accumulated lazily in
// 64 bits (one IMAD.WIDE per slot) and reduced once per block instead of four full Barrett rounds per slot and item.
__global__ void __launch_bounds__(RBS, 4) k_aggv_partial(ModQ m, StageConstF scf, const NttTables* __restrict__ tab,
                                                         const uint16_t* __restrict__ vk_ntt,
                                                         const int16_t* __restrict__ ch_pairs, int ch_wt,
                                                         const int16_t* __restrict__ ag_pairs, int64_t count,
                                                         int32_t* __restrict__ partial) {
    __shared__ __align__(16) uint32_t xbuf[(RBS / 32) * XWARP];
    __shared__ __align__(16) uint4 twtab[LANES * TW_ROW];
    __shared__ uint32_t pw[512];
    __shared__ uint32_t red[D];
    for (int i = threadIdx.x; i < 512; i += blockDim.x) pw[i] = tab->pw[i];
    for (int i = threadIdx.x; i < D; i += blockDim.x) red[i] = 0;
    fill_tw_shared(twtab, tab);
    const HalfWarp h = half_warp(xbuf);
    const LaneTwFShared twf{twtab + h.lane * TW_ROW};
    uint32_t odd[EPT];
#pragma unroll
    for (int k = 0; k < EPT; ++k) odd[k] = 2 * (__brev((uint32_t)(16 * h.lane + k)) >> 24) + 1;
    uint64_t acc[EPT];
#pragma unroll
    for (int k = 0; k < EPT; ++k) acc[k] = 0;
    const uint32_t* ap = reinterpret_cast<const uint32_t*>(ag_pairs);
    const uint32_t* cp = reinterpret_cast<const uint32_t*>(ch_pairs);
    // The first two challenge words of a lane (all of them for ch_wt <= 32) and the aggregation coefficient of the NEXT
    // item are requested one iteration ahead, the key rows at the top of the iteration: no global round trip is left
    // on the critical path of an item.
    const int64_t step = (int64_t)gridDim.x * HWB;
    auto item_of = [&](int64_t base) { const int64_t raw = base + h.slot; return raw < count ? raw : count - 1; };
    uint32_t n_c0 = 0, n_c1 = 0, n_pr = 0;
    auto prefetch = [&](int64_t base) {
        const int64_t it = item_of(base);
        const uint32_t* q = cp + it * ch_wt;
        n_c0 = h.lane < ch_wt ? __ldg(q + h.lane) : 0xFFFF0000u;            // index 0, coefficient -1: never written
        n_c1 = h.lane + LANES < ch_wt ? __ldg(q + h.lane + LANES) : 0xFFFF0000u;
        n_pr = __ldg(ap + it);
    };
    int64_t base = (int64_t)blockIdx.x * HWB;
    if (base < count) prefetch(base);
    for (; base < count; base += step) {
        const bool live = base + h.slot < count;
        const int64_t item = item_of(base);
        const uint32_t c0 = n_c0, c1 = n_c1, pr = n_pr;
        const uint4* vkp = reinterpret_cast<const uint4*>(vk_ntt + item * 2 * D + 16 * h.lane);
        const uint4 va = __ldg(vkp), vb = __ldg(vkp + 1), vc = __ldg(vkp + D / 8), vd = __ldg(vkp + D / 8 + 1);
        if (base + step < count) prefetch(base + step);
        uint32_t c[EPT];
        {
            int cx[EPT];
#pragma unroll
            for (int j = 0; j < EPT; ++j) h.xb[XROW * j + h.lane] = 0;
            __syncwarp();
            if (h.lane < ch_wt) h.xb[XROW * ((c0 & 0xFFu) >> 4) + (c0 & 15u)] = (uint32_t)(int)(int16_t)(c0 >> 16);
            if (h.lane + LANES < ch_wt) h.xb[XROW * ((c1 & 0xFFu) >> 4) + (c1 & 15u)] = (uint32_t)(int)(int16_t)(c1 >> 16);
            for (int e = h.lane + 2 * LANES; e < ch_wt; e += LANES) {
                const uint32_t w = __ldg(cp + item * ch_wt + e);
                h.xb[XROW * ((w & 0xFFu) >> 4) + (w & 15u)] = (uint32_t)(int)(int16_t)(w >> 16);
            }
            __syncwarp();
#pragma unroll
            for (int j = 0; j < EPT; ++j) cx[j] = (int)h.xb[XROW * j + h.lane];
            __syncwarp();
            ntt_fwd_256_fp(cx, c, m, scf, twf, h.xb, h.lane);
        }
        const uint32_t wl[8] = {va.x, va.y, va.z, va.w, vb.x, vb.y, vb.z, vb.w};
        const uint32_t wr[8] = {vc.x, vc.y, vc.z, vc.w, vd.x, vd.y, vd.z, vd.w};
        const uint32_t kk = pr & 0xFF;
        const uint32_t negoff = (int16_t)(pr >> 16) < 0 ? 256u : 0u;
#pragma unroll
        for (int k = 0; k < EPT; ++k) {
            const uint32_t vl = (k & 1) ? wl[k >> 1] >> 16 : wl[k >> 1] & 0xFFFFu;
            const uint32_t vr = (k & 1) ? wr[k >> 1] >> 16 : wr[k >> 1] & 0xFFFFu;
            uint32_t ck = barrett_lazy(c[k] - FP_BIAS, m);                 // < 2q
            ck = min(ck, ck - m.q);                                       // < q: the product below stays under 2^32
            const uint32_t t = barrett_lazy(ck * vl, m) + vr;             // < 2q + 2^16
            const uint32_t w = live ? pw[(odd[k] * kk + negoff) & 511] : 0u;
            acc[k] += (uint64_t)t * w;
        }
    }
#pragma unroll
    for (int k = 0; k < EPT; ++k) atomicAdd(&red[16 * h.lane + k], reduce64(acc[k], m));
    __syncthreads();
    for (int i = threadIdx.x; i < D; i += blockDim.x) atomicAdd(&partial[i], (int32_t)(red[i] % m.q));
}

// ------------------------------------------------------------------------------------------------
// Batches of independent aggregates (lcb_bklm_aggregate_batch / lcb_bklm_aggregate_verify_batch).  The sorted items of
// all groups lie back to back; gid[i] is the group of item i.  Each warp (half-warp) owns ONE CONTIGUOUS range of
// items, accumulates while consecutive items belong to the same group and flushes the sum into that group's slice of
// `partial` with atomicAdd when the group changes and at the end of its range.  A group is thus flushed at most once
// per warp (half-warp) whose range it touches, and each flush adds a value reduced mod q (|v| < q < 2^16): with at
// most SEG_MAX_WARPS such ranges per polynomial, |partial| < 2^14 * 2^16 = 2^30 and int32 cannot overflow.
constexpr int SEG_MAX_WARPS = 1 << 14;
// rows accumulated between in-register reductions of k_agg_partial_seg: 2^15 rows of |x| <= 2^15 stay below 2^30
constexpr int SEG_REDUCE_ROWS = 1 << 15;

// Aggregate: partial[g][i][p] += s * sig[t][i][(p - k) mod 256] * (p < k ? -1 : 1) over the items t of group g.
// grid = (chunks, l) as k_agg_partial, but warp w of polynomial i walks rows [w R, (w + 1) R) in order.  Rows are
// parked as E = [~row | row] exactly as in k_agg_partial; the wrapped reads (~v = -v - 1 instead of -v) are repaired
// per group: lane 0 counts s per rotation k in the warp's own histogram, and a flush adds
// corr[p] = sum over k > p of hist[k] (a warp suffix scan of the 256 counts) before it clears the histogram.
// Three resident blocks (79 registers); at four the 64-register cap spills 48 bytes.
// SIG_BITS = 0: int16 signatures.  SIG_BITS = 11 / 13: rows of the packed wire format (wire.cu; bias sig_bias), 22 / 26
// of the 32 lanes fetch 16 bytes of a row; at parking time the raw row goes to the lower half of its E buffer and every
// lane decodes its 8 values from there, so the fold below sees exactly the int16 row k_unpack would have made.
template <int SIG_BITS>
__global__ void __launch_bounds__(32 * AGG_WARPS, 3) k_agg_partial_seg(ModQ m, int l, const int16_t* __restrict__ sigs,
                                                                   const int16_t* __restrict__ ag_pairs,
                                                                   const int32_t* __restrict__ gid, int64_t total,
                                                                   int64_t n_agg, int64_t per_warp,
                                                                   int32_t* __restrict__ partial, int sig_bias) {
    constexpr int ROW_BYTES = SIG_BITS ? 32 * SIG_BITS : D * 2;
    __shared__ __align__(16) int32_t hist[AGG_WARPS][D];
    __shared__ __align__(16) int16_t rows[AGG_WARPS][AGG_DEPTH][2 * D];
    const int poly = blockIdx.y;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    int32_t* hw = hist[warp];
#pragma unroll
    for (int jj = 0; jj < 8; ++jj) hw[lane + 32 * jj] = 0;
    const int64_t t_begin = ((int64_t)blockIdx.x * AGG_WARPS + warp) * per_warp;
    const int64_t t_end = min(t_begin + per_warp, total);
    int left = t_begin < t_end ? (int)(t_end - t_begin) : 0;
    const uint32_t* app = reinterpret_cast<const uint32_t*>(ag_pairs) + t_begin;
    const int32_t* gp = gid + t_begin;
    const unsigned char* rowp = reinterpret_cast<const unsigned char*>(sigs) + (t_begin * l + poly) * ROW_BYTES + 16 * lane;
    const int64_t rstep = (int64_t)l * ROW_BYTES;
    int32_t acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    uint4 v[AGG_DEPTH];
    uint32_t pr[AGG_DEPTH];
    int grp[AGG_DEPTH];
    auto fetch = [&]() {                         // the next min(left, AGG_DEPTH) rows; missing rows are never folded
#pragma unroll
        for (int j = 0; j < AGG_DEPTH; ++j)
            if (j < left) {
                if (SIG_BITS == 0 || 16 * lane < ROW_BYTES)
                    v[j] = __ldg(reinterpret_cast<const uint4*>(rowp + j * rstep));
                pr[j] = __ldg(app + j);
                grp[j] = __ldg(gp + j);
            }
        LCB_CHECK(left <= 0 || (app - reinterpret_cast<const uint32_t*>(ag_pairs)) + min(left, AGG_DEPTH) <= total);
        rowp += AGG_DEPTH * rstep;
        app += AGG_DEPTH;
        gp += AGG_DEPTH;
    };
    int cur_g = -1, since = 0;
    auto flush = [&]() {
        __syncwarp();
        // corr[p] = sum_{k > p} hist[k]: lane owns counts 8 lane .. 8 lane + 7, suffix sums inside, then across lanes
        int4 h0 = *reinterpret_cast<const int4*>(hw + 8 * lane), h1 = *reinterpret_cast<const int4*>(hw + 8 * lane + 4);
        int hv[8] = {h0.x, h0.y, h0.z, h0.w, h1.x, h1.y, h1.z, h1.w};
        int sfx[8];
        sfx[7] = 0;
#pragma unroll
        for (int i = 6; i >= 0; --i) sfx[i] = sfx[i + 1] + hv[i + 1];
        const int own = sfx[0] + hv[0];
        int above = own;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int y = __shfl_down_sync(0xFFFFFFFFu, above, o);
            if (lane + o < 32) above += y;
        }
        above -= own;
        __syncwarp();
        *reinterpret_cast<int4*>(hw + 8 * lane) = make_int4(sfx[0] + above, sfx[1] + above, sfx[2] + above, sfx[3] + above);
        *reinterpret_cast<int4*>(hw + 8 * lane + 4) = make_int4(sfx[4] + above, sfx[5] + above, sfx[6] + above, sfx[7] + above);
        __syncwarp();
        LCB_CHECK(cur_g >= 0 && cur_g < n_agg);
        int32_t* out = partial + ((int64_t)cur_g * l + poly) * D;
#pragma unroll
        for (int jj = 0; jj < 8; ++jj) {
            // |acc| < q + 2^30 and |corr| <= 2^30 before the reduction of corr: no int32 overflow
            const int32_t r = (acc[jj] + hw[lane + 32 * jj] % (int)m.q) % (int)m.q;
            atomicAdd(out + lane + 32 * jj, r);
            acc[jj] = 0;
        }
        __syncwarp();
#pragma unroll
        for (int jj = 0; jj < 8; ++jj) hw[lane + 32 * jj] = 0;
        __syncwarp();
        since = 0;
    };
    if (left > 0) fetch();
    const unsigned rows_s = (unsigned)__cvta_generic_to_shared(rows[warp][0]);
    while (left > 0) {
        const int nrow = min(left, AGG_DEPTH);
        uint32_t cur[AGG_DEPTH];
        int cg[AGG_DEPTH];
        __syncwarp();
        if constexpr (SIG_BITS != 0) {
            // value 8 lane + i sits at bit (8 lane + i) * SIG_BITS of the row; the word after the last one read lies
            // inside the 1 KB E buffer and only contributes bits the mask drops
#pragma unroll
            for (int j = 0; j < AGG_DEPTH; ++j)
                if (16 * lane < ROW_BYTES) reinterpret_cast<uint4*>(rows[warp][j])[lane] = v[j];
            __syncwarp();
#pragma unroll
            for (int j = 0; j < AGG_DEPTH; ++j) {
                const uint32_t* rw = reinterpret_cast<const uint32_t*>(rows[warp][j]);
                uint32_t w[4];
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    const int pos = (8 * lane + i) * SIG_BITS;
                    const uint32_t f = __funnelshift_r(rw[pos >> 5], rw[(pos >> 5) + 1], pos & 31) & ((1u << SIG_BITS) - 1);
                    const uint32_t x = (f - (uint32_t)sig_bias) & 0xFFFFu;
                    if (i & 1) w[i >> 1] |= x << 16;
                    else w[i >> 1] = x;
                }
                v[j] = make_uint4(w[0], w[1], w[2], w[3]);
            }
            __syncwarp();
        }
#pragma unroll
        for (int j = 0; j < AGG_DEPTH; ++j) {
            uint4* e = reinterpret_cast<uint4*>(rows[warp][j]);
            e[lane] = make_uint4(~v[j].x, ~v[j].y, ~v[j].z, ~v[j].w);
            e[32 + lane] = v[j];
            cur[j] = pr[j];
            cg[j] = grp[j];
        }
        __syncwarp();
        left -= AGG_DEPTH;
        if (left > 0) fetch();                   // next rows in flight while this batch is folded
#pragma unroll
        for (int j = 0; j < AGG_DEPTH; ++j) {
            if (j < nrow) {                      // warp-uniform
                if (cg[j] != cur_g) {
                    if (cur_g >= 0) flush();
                    cur_g = cg[j];
                } else if (since == SEG_REDUCE_ROWS) {
#pragma unroll
                    for (int jj = 0; jj < 8; ++jj) acc[jj] %= (int)m.q;
                    since = 0;
                }
                const int k = (int)(cur[j] & 0xFF);
                const int sg = (int)(int16_t)(cur[j] >> 16);
                const unsigned a = rows_s + (unsigned)(j * 4 * D) + 2u * (unsigned)(D - k + lane);
#pragma unroll
                for (int jj = 0; jj < 8; ++jj) {
                    int x;
                    asm volatile("ld.shared.s16 %0, [%1];" : "=r"(x) : "r"(a + 64u * jj));
                    acc[jj] += sg * x;
                }
                if (lane == 0) hw[k] += sg;
                ++since;
            }
        }
    }
    if (cur_g >= 0) flush();
}

// Aggregate-verify right-hand sides of many groups: the per-item math of k_aggv_partial (one half-warp per item,
// FP32-assisted challenge transform, lazy 64-bit accumulation), but half-warp h walks items [h R, (h + 1) R) in order
// and flushes per group.  Every half-warp runs the same number of trips (items past its range are dead, as the clamped
// tail of k_aggv_partial) because the transform synchronises the whole warp.  A trip adds t * w < 2^18 * 2^16 to the
// accumulator; reduce64 takes sums below 2^54, so a range holds at most 2^20 items (the launcher sizes the grid so).
// VK_BITS = 0: uint16 key slots (also the 16-bit wire format, whose bytes are that array); VK_BITS = 14: keys in the
// 14-bit wire format, 7 words per lane and key half, expanded as k_verify<..., 14> does.
template <int VK_BITS>
__global__ void __launch_bounds__(RBS, 4) k_aggv_partial_seg(ModQ m, StageConstF scf, const NttTables* __restrict__ tab,
                                                             const uint16_t* __restrict__ vk_ntt,
                                                             const int16_t* __restrict__ ch_pairs, int ch_wt,
                                                             const int16_t* __restrict__ ag_pairs,
                                                             const int32_t* __restrict__ gid, int64_t total,
                                                             int64_t n_agg, int64_t per_hw, int32_t* __restrict__ partial) {
    __shared__ __align__(16) uint32_t xbuf[(RBS / 32) * XWARP];
    __shared__ __align__(16) uint4 twtab[LANES * TW_ROW];
    __shared__ uint32_t pw[512];
    for (int i = threadIdx.x; i < 512; i += blockDim.x) pw[i] = tab->pw[i];
    fill_tw_shared(twtab, tab);
    const HalfWarp h = half_warp(xbuf);
    const LaneTwFShared twf{twtab + h.lane * TW_ROW};
    uint32_t odd[EPT];
#pragma unroll
    for (int k = 0; k < EPT; ++k) odd[k] = 2 * (__brev((uint32_t)(16 * h.lane + k)) >> 24) + 1;
    uint64_t acc[EPT];
#pragma unroll
    for (int k = 0; k < EPT; ++k) acc[k] = 0;
    const uint32_t* ap = reinterpret_cast<const uint32_t*>(ag_pairs);
    const uint32_t* cp = reinterpret_cast<const uint32_t*>(ch_pairs);
    const int64_t t_begin = ((int64_t)blockIdx.x * HWB + h.slot) * per_hw;
    const int64_t t_end = min(t_begin + per_hw, total);
    auto item_of = [&](int64_t t) { return t < t_end ? t : (t_begin < total ? t_begin : total - 1); };
    uint32_t n_c0 = 0, n_c1 = 0, n_pr = 0;
    int n_g = 0;
    auto prefetch = [&](int64_t t) {
        const int64_t it = item_of(t);
        LCB_CHECK(it >= 0 && it < total);
        const uint32_t* q = cp + it * ch_wt;
        n_c0 = h.lane < ch_wt ? __ldg(q + h.lane) : 0xFFFF0000u;            // index 0, coefficient -1: never written
        n_c1 = h.lane + LANES < ch_wt ? __ldg(q + h.lane + LANES) : 0xFFFF0000u;
        n_pr = __ldg(ap + it);
        n_g = __ldg(gid + it);
    };
    int cur_g = -1;
    auto flush = [&]() {
        LCB_CHECK(cur_g >= 0 && cur_g < n_agg);
#pragma unroll
        for (int k = 0; k < EPT; ++k) {
            atomicAdd(&partial[(int64_t)cur_g * D + 16 * h.lane + k], (int32_t)reduce64(acc[k], m));
            acc[k] = 0;
        }
    };
    prefetch(t_begin);
    for (int64_t t = t_begin; t < t_begin + per_hw; ++t) {
        const bool live = t < t_end;
        const int64_t item = item_of(t);
        const uint32_t c0 = n_c0, c1 = n_c1, pr = n_pr;
        const int g = n_g;
        uint4 va, vb, vc, vd;
        if constexpr (VK_BITS == 14) {
            LCB_CHECK(item >= 0 && item < total);
            const uint32_t* vkp = reinterpret_cast<const uint32_t*>(vk_ntt) + item * (2 * 112) + 7 * h.lane;
            va = make_uint4(__ldg(vkp), __ldg(vkp + 1), __ldg(vkp + 2), __ldg(vkp + 3));
            vb = make_uint4(__ldg(vkp + 4), __ldg(vkp + 5), __ldg(vkp + 6), 0u);
            vc = make_uint4(__ldg(vkp + 112), __ldg(vkp + 113), __ldg(vkp + 114), __ldg(vkp + 115));
            vd = make_uint4(__ldg(vkp + 116), __ldg(vkp + 117), __ldg(vkp + 118), 0u);
        } else {
            const uint4* vkp = reinterpret_cast<const uint4*>(vk_ntt + item * 2 * D + 16 * h.lane);
            va = __ldg(vkp), vb = __ldg(vkp + 1), vc = __ldg(vkp + D / 8), vd = __ldg(vkp + D / 8 + 1);
        }
        if (t + 1 < t_begin + per_hw) prefetch(t + 1);
        uint32_t c[EPT];
        {
            int cx[EPT];
#pragma unroll
            for (int j = 0; j < EPT; ++j) h.xb[XROW * j + h.lane] = 0;
            __syncwarp();
            if (h.lane < ch_wt) h.xb[XROW * ((c0 & 0xFFu) >> 4) + (c0 & 15u)] = (uint32_t)(int)(int16_t)(c0 >> 16);
            if (h.lane + LANES < ch_wt) h.xb[XROW * ((c1 & 0xFFu) >> 4) + (c1 & 15u)] = (uint32_t)(int)(int16_t)(c1 >> 16);
            for (int e = h.lane + 2 * LANES; e < ch_wt; e += LANES) {
                const uint32_t w = __ldg(cp + item * ch_wt + e);
                h.xb[XROW * ((w & 0xFFu) >> 4) + (w & 15u)] = (uint32_t)(int)(int16_t)(w >> 16);
            }
            __syncwarp();
#pragma unroll
            for (int j = 0; j < EPT; ++j) cx[j] = (int)h.xb[XROW * j + h.lane];
            __syncwarp();
            ntt_fwd_256_fp(cx, c, m, scf, twf, h.xb, h.lane);
        }
        if (live && g != cur_g) {                // half-warp-uniform
            if (cur_g >= 0) flush();
            cur_g = g;
        }
        const uint32_t wl[8] = {va.x, va.y, va.z, va.w, vb.x, vb.y, vb.z, vb.w};
        const uint32_t wr[8] = {vc.x, vc.y, vc.z, vc.w, vd.x, vd.y, vd.z, vd.w};
        const uint32_t kk = pr & 0xFF;
        const uint32_t negoff = (int16_t)(pr >> 16) < 0 ? 256u : 0u;
#pragma unroll
        for (int k = 0; k < EPT; ++k) {
            uint32_t vl, vr;
            if constexpr (VK_BITS == 14) {
                vl = __funnelshift_r(wl[(14 * k) >> 5], wl[((14 * k) >> 5) + 1], (14 * k) & 31) & 0x3FFFu;
                vr = __funnelshift_r(wr[(14 * k) >> 5], wr[((14 * k) >> 5) + 1], (14 * k) & 31) & 0x3FFFu;
            } else {
                vl = (k & 1) ? wl[k >> 1] >> 16 : wl[k >> 1] & 0xFFFFu;
                vr = (k & 1) ? wr[k >> 1] >> 16 : wr[k >> 1] & 0xFFFFu;
            }
            uint32_t ck = barrett_lazy(c[k] - FP_BIAS, m);                 // < 2q
            ck = min(ck, ck - m.q);                                       // < q: the product below stays under 2^32
            const uint32_t tt = barrett_lazy(ck * vl, m) + vr;            // < 2q + 2^16
            const uint32_t w = live ? pw[(odd[k] * kk + negoff) & 511] : 0u;
            acc[k] += (uint64_t)tt * w;
        }
    }
    if (cur_g >= 0) flush();
}

// partial int32[n][256] -> residues uint16 in [0, q): the right-hand sides k_verify compares key_ch * ag_sig with
__global__ void k_aggv_residues(ModQ m, const int32_t* __restrict__ partial, int64_t nelem, uint16_t* __restrict__ out) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nelem; i += (int64_t)gridDim.x * blockDim.x) {
        int v = partial[i] % (int)m.q;
        out[i] = (uint16_t)(v < 0 ? v + (int)m.q : v);
    }
}

// The lower limits k_verify does not test: 1 <= count_g <= ag_cap and ag_sig[g] != 0 (max |coefficient| >= 1, i.e. also
// weight >= 1).  One thread per group; the zero test stops at the first non-zero 16 bytes, so an honest aggregate costs
// one sector and the aggregate signatures are not read a second time.
__global__ void k_aggv_limits(const int64_t* __restrict__ agg_off, int64_t n_agg, const int16_t* __restrict__ ag_sig,
                              int64_t words16, int64_t ag_cap, uint8_t* __restrict__ verdict) {
    for (int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; g < n_agg; g += (int64_t)gridDim.x * blockDim.x) {
        if (!verdict[g]) continue;
        const int64_t cnt = __ldg(agg_off + g + 1) - __ldg(agg_off + g);
        bool ok = cnt >= 1 && cnt <= ag_cap;
        if (ok) {
            const uint4* p = reinterpret_cast<const uint4*>(ag_sig) + g * words16;
            bool nz = false;
            for (int64_t w = 0; w < words16 && !nz; ++w) {
                const uint4 x = __ldg(p + w);
                nz = (x.x | x.y | x.z | x.w) != 0;
            }
            ok = nz;
        }
        if (!ok) verdict[g] = 0;
    }
}

// The same on packed aggregates (wire.cu layout, `bits` bits per coefficient, bias `bias`): a coefficient is non-zero
// exactly where its field differs from the bias.  The test stops at the first such field.
__global__ void k_aggv_limits_packed(const int64_t* __restrict__ agg_off, int64_t n_agg, const uint32_t* __restrict__ ag_packed,
                                     int64_t fields, int bits, uint32_t bias, int64_t ag_cap, uint8_t* __restrict__ verdict) {
    const int64_t words = fields * bits / 32;          // fields = l * 256: whole words
    const uint32_t mask = (1u << bits) - 1;
    for (int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; g < n_agg; g += (int64_t)gridDim.x * blockDim.x) {
        if (!verdict[g]) continue;
        const int64_t cnt = __ldg(agg_off + g + 1) - __ldg(agg_off + g);
        bool ok = cnt >= 1 && cnt <= ag_cap;
        if (ok) {
            const uint32_t* p = ag_packed + g * words;
            bool nz = false;
            for (int64_t i = 0; i < fields && !nz; ++i) {
                const int64_t pos = i * bits, w = pos >> 5;
                LCB_CHECK(w < words);
                const uint32_t hi = w + 1 < words ? __ldg(p + w + 1) : 0u;
                nz = (__funnelshift_r(__ldg(p + w), hi, (unsigned)pos & 31u) & mask) != bias;
            }
            ok = nz;
        }
        if (!ok) verdict[g] = 0;
    }
}

// bounds on ag_sig (with lower limits), key_ch * ag_sig == partial sum; one half-warp
__global__ void __launch_bounds__(32) k_aggv_finish(ModQ m, StageConst sc, const NttTables* __restrict__ tab,
                                                    const uint32_t* __restrict__ a_hat, int l,
                                                    const int32_t* __restrict__ partial,
                                                    const int16_t* __restrict__ ag_sig, int64_t total, int ag_cap,
                                                    int avf_bd, int avf_wt, uint8_t* __restrict__ verdict) {
    __shared__ __align__(16) uint32_t xbuf[XWARP];
    const HalfWarp h = half_warp(xbuf);
    LaneTw tw;
    load_lane_tw(tw, tab->w, tab->ws, h.lane);
    uint64_t acc[EPT];
#pragma unroll
    for (int i = 0; i < EPT; ++i) acc[i] = 0;
    int maxabs = 0, maxw = 0;
    for (int i = 0; i < l; ++i) {
        const int16_t* p = ag_sig + i * D;
        uint32_t r[EPT];
        int nz = 0;
#pragma unroll
        for (int j = 0; j < EPT; ++j) {
            int x = __ldg(p + h.lane + 16 * j);
            maxabs = max(maxabs, abs(x));
            nz += (x != 0);
            r[j] = (uint32_t)(x + (int)m.cq);
        }
#pragma unroll
        for (int o = 8; o >= 1; o >>= 1) nz += __shfl_xor_sync(0xFFFFFFFFu, nz, o);
        maxw = max(maxw, nz);
        ntt_fwd_256(r, m, sc, tw, h.xb, h.lane);
#pragma unroll
        for (int g = 0; g < EPT; ++g) acc[g] += (uint64_t)r[g] * __ldg(a_hat + i * D + 16 * h.lane + g);
    }
#pragma unroll
    for (int o = 8; o >= 1; o >>= 1) maxabs = max(maxabs, __shfl_xor_sync(0xFFFFFFFFu, maxabs, o));
    bool ok = maxabs >= 1 && maxabs <= avf_bd && maxw >= 1 && maxw <= avf_wt && total >= 1 && total <= ag_cap;
#pragma unroll
    for (int k = 0; k < EPT; ++k) {
        int v = partial[16 * h.lane + k] % (int)m.q;
        if (v < 0) v += (int)m.q;
        ok &= reduce64(acc[k], m) == (uint32_t)v;
    }
    const unsigned votes = __ballot_sync(0xFFFFFFFFu, ok);
    if (threadIdx.x == 0) verdict[0] = (votes & 0xFFFFu) == 0xFFFFu ? 1 : 0;
}

// ------------------------------------------------------------------------------------------------
template <typename K>
int resident_blocks(K kernel, int threads, size_t smem) {
    int nb = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, kernel, threads, smem) != cudaSuccess || nb < 1) nb = 1;
    return nb;
}

inline unsigned persistent_grid(int64_t items, int per_block, int num_sms, int resident) {
    int64_t need = (items + per_block - 1) / per_block;
    int64_t cap = (int64_t)num_sms * resident;
    return (unsigned)(need < cap ? need : cap);
}

inline size_t ring_smem(int l, int threads = RBS) { return (size_t)l * AROW * 4 + (size_t)(threads / 32) * XWARP * 4; }
// a_hat + transposition buffers + stage buffers + twiddle table (k_matvec; k_verify adds its 16 x 16 correction table)
inline size_t matvec_smem(int l) { return ring_smem(l, MBS) + (size_t)MHWB * STAGE_HALF_BYTES + (size_t)TW_BYTES; }
inline size_t verify_smem(int l) {
    return ring_smem(l, VBS) + (size_t)VHWB * STAGE_HALF_BYTES + (size_t)TW_BYTES + (size_t)LANES * EPT * 4;
}

template <typename K>
cudaError_t allow_smem(K kernel, size_t smem) {
    return cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
}

}  // namespace

cudaError_t launch_ntt_fwd(const RingCtx& c, const int16_t* coef, int64_t npoly, uint16_t* out, cudaStream_t st) {
    if (npoly <= 0) return cudaSuccess;
    unsigned grid = persistent_grid(npoly, HWB, c.num_sms, resident_blocks(k_ntt_fwd, RBS, 0));
    k_ntt_fwd<<<grid, RBS, 0, st>>>(c.m, c.sc, c.tab, coef, npoly, out);
    return cudaGetLastError();
}

cudaError_t launch_ntt_ref_repr(const RingCtx& c, const int16_t* coef, int64_t npoly, int16_t* out, cudaStream_t st) {
    if (npoly <= 0) return cudaSuccess;
    unsigned grid = persistent_grid(npoly, HWB, c.num_sms, resident_blocks(k_ntt_ref_repr, RBS, 0));
    k_ntt_ref_repr<<<grid, RBS, 0, st>>>(c.m, c.sc, c.tab, coef, npoly, out);
    return cudaGetLastError();
}

cudaError_t launch_ntt_inv(const RingCtx& c, const uint16_t* in, int64_t npoly, int16_t* coef, cudaStream_t st) {
    if (npoly <= 0) return cudaSuccess;
    unsigned grid = persistent_grid(npoly, HWB, c.num_sms, resident_blocks(k_ntt_inv, RBS, 0));
    k_ntt_inv<<<grid, RBS, 0, st>>>(c.m, c.sc, c.tab, in, npoly, coef);
    return cudaGetLastError();
}

cudaError_t launch_poly_mul(const RingCtx& c, const int16_t* a, const int16_t* b, int64_t npoly, int16_t* out,
                            cudaStream_t st) {
    if (npoly <= 0) return cudaSuccess;
    unsigned grid = persistent_grid(npoly, HWB, c.num_sms, resident_blocks(k_poly_mul, RBS, 0));
    k_poly_mul<<<grid, RBS, 0, st>>>(c.m, c.sc, c.tab, a, b, npoly, out);
    return cudaGetLastError();
}

cudaError_t launch_matvec(const RingCtx& c, const int16_t* vec_coef, int64_t nvec, uint16_t* vec_ntt,
                          uint16_t* y_ntt, int16_t* y_coef, cudaStream_t st) {
    if (nvec <= 0) return cudaSuccess;
    size_t smem = matvec_smem(c.l);
    cudaError_t e = allow_smem(k_matvec, smem);
    if (e != cudaSuccess) return e;
    unsigned grid = persistent_grid(nvec, MHWB, c.num_sms, resident_blocks(k_matvec, MBS, smem));
    k_matvec<<<grid, MBS, smem, st>>>(c.m, c.sc, c.scf, c.tab, c.a_hat, c.l, vec_coef, nvec, vec_ntt, y_ntt, y_coef);
    return cudaGetLastError();
}

template <int SIG_BITS>
cudaError_t launch_sign_t(const RingCtx& c, const uint16_t* sk_ntt, const int16_t* ch_pairs, int ch_wt, int64_t n,
                          void* sig, uint8_t* in_range, int sig_bias, cudaStream_t st) {
    if (n <= 0) return cudaSuccess;
    const size_t smem = (size_t)(RBS / 32) * XWARP * 4 + (size_t)HWB * SIGN_STAGE_BYTES + (size_t)TW_BYTES + (size_t)ITW_BYTES;
    cudaError_t e = allow_smem(k_sign<SIG_BITS>, smem);
    if (e != cudaSuccess) return e;
    unsigned grid = persistent_grid(n, HWB, c.num_sms, resident_blocks(k_sign<SIG_BITS>, RBS, smem));
    k_sign<SIG_BITS><<<grid, RBS, smem, st>>>(c.m, c.scf, c.iscf, c.tab, c.l, sk_ntt, ch_pairs, ch_wt, n,
                                              static_cast<int16_t*>(sig), in_range, sig_bias);
    return cudaGetLastError();
}

cudaError_t launch_sign(const RingCtx& c, const uint16_t* sk_ntt, const int16_t* ch_pairs, int ch_wt, int64_t n,
                        int16_t* sig, cudaStream_t st) {
    return launch_sign_t<0>(c, sk_ntt, ch_pairs, ch_wt, n, sig, nullptr, 0, st);
}

// The two shipped signature widths are written by k_sign itself; anything else is reported as unsupported and the
// caller signs into int16 scratch and packs.
cudaError_t launch_sign_packed(const RingCtx& c, const uint16_t* sk_ntt, const int16_t* ch_pairs, int ch_wt, int64_t n,
                               int sig_bits, int sig_bias, uint8_t* sig_packed, uint8_t* in_range, cudaStream_t st) {
    if (sig_bits == 11) return launch_sign_t<11>(c, sk_ntt, ch_pairs, ch_wt, n, sig_packed, in_range, sig_bias, st);
    if (sig_bits == 13) return launch_sign_t<13>(c, sk_ntt, ch_pairs, ch_wt, n, sig_packed, in_range, sig_bias, st);
    return cudaErrorNotSupported;
}

template <int SIG_BITS, int VK_BITS, int ST_BITS = 0, int RHS_BITS = 0>
cudaError_t launch_verify_t(const RingCtx& c, const void* vec, const void* vk, const int16_t* ch_pairs, int ch_wt,
                            const uint16_t* rhs_only, const uint16_t* extra_rhs, int64_t n, int bd, int wt, int sig_bias,
                            uint8_t* verdict, cudaStream_t st) {
    if (n <= 0) return cudaSuccess;
    if (n > ((int64_t)1 << 30)) return cudaErrorInvalidValue;      // 32-bit item indices inside the kernel
    size_t smem = verify_smem(c.l);
    auto kern = wt < D ? k_verify<true, SIG_BITS, VK_BITS, ST_BITS, RHS_BITS> : k_verify<false, SIG_BITS, VK_BITS, ST_BITS, RHS_BITS>;
    cudaError_t e = allow_smem(kern, smem);
    if (e != cudaSuccess) return e;
    unsigned grid = persistent_grid(n, VHWB, c.num_sms, resident_blocks(kern, VBS, smem));
    kern<<<grid, VBS, smem, st>>>(c.m, c.sc, c.scf, c.tab, c.a_hat, c.l, static_cast<const int16_t*>(vec),
                                  static_cast<const uint16_t*>(vk), ch_pairs, ch_wt, rhs_only, extra_rhs, n, bd, wt,
                                  sig_bias, verdict);
    return cudaGetLastError();
}

cudaError_t launch_verify(const RingCtx& c, const int16_t* vec_coef, const uint16_t* vk_ntt, const int16_t* ch_pairs,
                          int ch_wt, const uint16_t* rhs_only, const uint16_t* extra_rhs, int64_t n, int bd, int wt,
                          uint8_t* verdict, cudaStream_t st) {
    if (n <= 0) return cudaSuccess;
    if (n > ((int64_t)1 << 30)) return cudaErrorInvalidValue;      // 32-bit item indices inside the kernel
    // k_verify_tc walks the 4 l chunks of a 128-verify tile one after the other: about 70 us for any batch up to one
    // tile per SM.  k_verify takes 27 us for one verify and grows by a trip of 32 verifies per SM: 66 us at 14,208
    // verifies, 82 us at 18,944, where k_verify_tc takes 72 us (B200, secpar 128).  Smaller batches, the single drop-in
    // verify among them, keep k_verify.
    if (n < (int64_t)TC_MIN_TILES_PER_SM * TC_ROWS * c.num_sms)
        return launch_verify_t<0, 0>(c, vec_coef, vk_ntt, ch_pairs, ch_wt, rhs_only, extra_rhs, n, bd, wt, 0, verdict, st);
    const size_t smem = tc_smem_bytes();
    const bool lazy = c.m.q <= 32768;
    auto kern = wt < D ? (lazy ? k_verify_tc<true, true> : k_verify_tc<true, false>)
                       : (lazy ? k_verify_tc<false, true> : k_verify_tc<false, false>);
    cudaError_t e = allow_smem(kern, smem);
    if (e != cudaSuccess) return e;
    const uint32_t q = c.m.q, zn = q - c.zeta;
    const uint64_t b15 = 32768 % q;                                // -> kz = -(32768 + 32768 z) mod q
    const uint32_t kz0 = (uint32_t)((2 * (uint64_t)q - b15 - b15 * c.zeta % q) % q);
    const uint32_t kz1 = (uint32_t)((2 * (uint64_t)q - b15 - b15 * zn % q) % q);
    const int64_t tiles = (n + TC_ROWS - 1) / TC_ROWS;
    const unsigned grid = (unsigned)(tiles < c.num_sms ? tiles : c.num_sms);
    kern<<<grid, TC_THREADS, smem, st>>>(c.m, c.scf, c.tab, c.tc_b, c.l, vec_coef, vk_ntt, ch_pairs, ch_wt, rhs_only,
                                          extra_rhs, n, bd, wt, c.zeta, kz0, kz1, verdict);
    return cudaGetLastError();
}

cudaError_t launch_verify_tc_matrix(const RingCtx& c, cudaStream_t st) {
    k_verify_tc_matrix<<<c.num_sms * 4, 256, 0, st>>>(c.m, c.tab, c.a_hat, c.l, c.tc_b);
    return cudaGetLastError();
}

// The two shipped packings are expanded inside the kernel; anything else is reported as unsupported and the
// caller unpacks first.
// Packed statements (adaptor verify) have the width of the keys: 14 bits are read by k_verify<..., 11, 14, 14>; 16-bit
// rows are uint16 rows, read as such.
cudaError_t launch_verify_packed(const RingCtx& c, const uint8_t* sig_packed, int sig_bits, int sig_bias,
                                 const uint8_t* vk_packed, int vk_bits, const int16_t* ch_pairs, int ch_wt, int64_t n,
                                 int bd, int wt, uint8_t* verdict, cudaStream_t st, const uint8_t* st_packed) {
    const uint16_t* ex = reinterpret_cast<const uint16_t*>(st_packed);
    if (sig_bits == 11 && vk_bits == 14 && st_packed)
        return launch_verify_t<11, 14, 14>(c, sig_packed, vk_packed, ch_pairs, ch_wt, nullptr, ex, n, bd, wt, sig_bias, verdict, st);
    if (sig_bits == 11 && vk_bits == 14)
        return launch_verify_t<11, 14>(c, sig_packed, vk_packed, ch_pairs, ch_wt, nullptr, nullptr, n, bd, wt, sig_bias, verdict, st);
    if (sig_bits == 13 && vk_bits == 16)
        return launch_verify_t<13, 0>(c, sig_packed, vk_packed, ch_pairs, ch_wt, nullptr, ex, n, bd, wt, sig_bias, verdict, st);
    return cudaErrorNotSupported;
}

// Witness-verify form on packed rows: BKLM aggregates (12 / 14 bits, uint16 right-hand sides) and adaptor witnesses with
// packed statements (witnesses 2 bits, or 12 / 14 as extracted; statements 14 or 16 bits, bias 0).  The decoder of
// k_verify is the one of the signature widths, and at even widths every value starts in the same half-word phase.  A
// 16-bit statement row has the bytes of a uint16 row; 14-bit rows are read by k_verify<..., RHS_BITS = 14>.
cudaError_t launch_verify_rhs_packed(const RingCtx& c, const uint8_t* vec_packed, int bits, int bias, const uint16_t* rhs_only,
                                     int64_t n, int bd, int wt, uint8_t* verdict, cudaStream_t st, int rhs_bits) {
    if (rhs_bits == 16 && bits == 12)
        return launch_verify_t<12, 0>(c, vec_packed, nullptr, nullptr, 0, rhs_only, nullptr, n, bd, wt, bias, verdict, st);
    if (rhs_bits == 16 && bits == 14)
        return launch_verify_t<14, 0>(c, vec_packed, nullptr, nullptr, 0, rhs_only, nullptr, n, bd, wt, bias, verdict, st);
    if (rhs_bits == 16 && bits == 2)
        return launch_verify_t<2, 0>(c, vec_packed, nullptr, nullptr, 0, rhs_only, nullptr, n, bd, wt, bias, verdict, st);
    if (rhs_bits == 14 && bits == 2)
        return launch_verify_t<2, 0, 0, 14>(c, vec_packed, nullptr, nullptr, 0, rhs_only, nullptr, n, bd, wt, bias, verdict, st);
    if (rhs_bits == 14 && bits == 12)
        return launch_verify_t<12, 0, 0, 14>(c, vec_packed, nullptr, nullptr, 0, rhs_only, nullptr, n, bd, wt, bias, verdict, st);
    return cudaErrorNotSupported;
}

cudaError_t launch_vec_addsub(const RingCtx& c, const int16_t* a, const int16_t* b, int64_t nelem, int sub,
                              int16_t* out, cudaStream_t st) {
    if (nelem <= 0) return cudaSuccess;
    int64_t need = (nelem / 8 + 255) / 256;
    int64_t cap = (int64_t)c.num_sms * 8;
    k_vec_addsub<<<(unsigned)(need < cap ? need : cap), 256, 0, st>>>(c.m, a, b, nelem, sub, out);
    return cudaGetLastError();
}

cudaError_t launch_agg_partial(const RingCtx& c, const int16_t* sigs, const int16_t* ag_pairs, int64_t count,
                               int32_t* partial, cudaStream_t st) {
    if (count <= 0) return cudaSuccess;
    const int64_t per_block = (int64_t)AGG_WARPS * AGG_DEPTH;          // one batch of rows per warp
    int64_t need = (count + per_block - 1) / per_block;
    // exactly one resident wave: chunks * l blocks <= SMs * resident blocks
    int64_t cap = (int64_t)c.num_sms * resident_blocks(k_agg_partial, 32 * AGG_WARPS, 0) / c.l;
    if (cap < 1) cap = 1;
    dim3 grid((unsigned)(need < cap ? need : cap), (unsigned)c.l);
    k_agg_partial<<<grid, 32 * AGG_WARPS, 0, st>>>(c.m, c.l, sigs, ag_pairs, count, partial);
    return cudaGetLastError();
}

cudaError_t launch_agg_finish(const RingCtx& c, const int32_t* partial, int16_t* ag_sig, cudaStream_t st) {
    int n = c.l * D;
    k_agg_finish<<<(n + 255) / 256, 256, 0, st>>>(c.m, partial, n, ag_sig);
    return cudaGetLastError();
}

cudaError_t launch_aggv_partial(const RingCtx& c, const uint16_t* vk_ntt, const int16_t* ch_pairs, int ch_wt,
                                const int16_t* ag_pairs, int64_t count, int32_t* partial, cudaStream_t st) {
    if (count <= 0) return cudaSuccess;
    unsigned grid = persistent_grid(count, HWB, c.num_sms, resident_blocks(k_aggv_partial, RBS, 0));
    k_aggv_partial<<<grid, RBS, 0, st>>>(c.m, c.scf, c.tab, vk_ntt, ch_pairs, ch_wt, ag_pairs, count, partial);
    return cudaGetLastError();
}

cudaError_t launch_aggv_finish(const RingCtx& c, const int32_t* partial, const int16_t* ag_sig, int64_t total,
                               int ag_cap, int avf_bd, int avf_wt, uint8_t* verdict, cudaStream_t st) {
    k_aggv_finish<<<1, 32, 0, st>>>(c.m, c.sc, c.tab, c.a_hat, c.l, partial, ag_sig, total, ag_cap, avf_bd, avf_wt,
                                    verdict);
    return cudaGetLastError();
}

cudaError_t launch_agg_finish_n(const RingCtx& c, const int32_t* partial, int64_t nelem, int16_t* ag_sig, cudaStream_t st) {
    // k_agg_finish indexes with int: chunks of 2^30 elements
    for (int64_t first = 0; first < nelem; first += (int64_t)1 << 30) {
        const int n = (int)min(nelem - first, (int64_t)1 << 30);
        k_agg_finish<<<(n + 255) / 256, 256, 0, st>>>(c.m, partial + first, n, ag_sig + first);
        cudaError_t e = cudaGetLastError();
        if (e != cudaSuccess) return e;
    }
    return cudaSuccess;
}

// Test knob LCB_SEG_RANGES: an upper limit on the ranges (warps / half-warps) per polynomial of the segmented kernels, so
// that tests reach long ranges - in-register reductions, many flushes per range - without gigabytes of input.  It can
// only lower the computed count; values below 1 are ignored.
static int64_t seg_ranges(int64_t ranges) {
    if (const char* env = getenv("LCB_SEG_RANGES")) {
        const int64_t v = atoll(env);
        if (v >= 1 && v < ranges) return v;
    }
    return ranges;
}

cudaError_t launch_agg_partial_seg(const RingCtx& c, const void* sigs, int sig_bits, int sig_bias, const int16_t* ag_pairs,
                                   const int32_t* gid, int64_t total, int64_t n_agg, int32_t* partial, cudaStream_t st) {
    if (total <= 0) return cudaSuccess;
    if (sig_bits != 0 && sig_bits != 11 && sig_bits != 13) return cudaErrorNotSupported;
    auto kern = sig_bits == 11 ? k_agg_partial_seg<11> : sig_bits == 13 ? k_agg_partial_seg<13> : k_agg_partial_seg<0>;
    int64_t cap = (int64_t)c.num_sms * resident_blocks(kern, 32 * AGG_WARPS, 0) / c.l;
    cap = max((int64_t)1, min(cap, (int64_t)SEG_MAX_WARPS / AGG_WARPS));
    const int64_t need = (total + AGG_WARPS * AGG_DEPTH - 1) / (AGG_WARPS * AGG_DEPTH);
    const int64_t ranges = seg_ranges(min(need, cap) * AGG_WARPS);      // warps past the last range find nothing to do
    const int64_t chunks = (ranges + AGG_WARPS - 1) / AGG_WARPS;
    const int64_t per_warp = (total + ranges - 1) / ranges;
    dim3 grid((unsigned)chunks, (unsigned)c.l);
    kern<<<grid, 32 * AGG_WARPS, 0, st>>>(c.m, c.l, static_cast<const int16_t*>(sigs), ag_pairs, gid, total, n_agg, per_warp,
                                          partial, sig_bias);
    return cudaGetLastError();
}

cudaError_t launch_aggv_partial_seg(const RingCtx& c, const void* vk_ntt, int vk_bits, const int16_t* ch_pairs, int ch_wt,
                                    const int16_t* ag_pairs, const int32_t* gid, int64_t total, int64_t n_agg,
                                    int32_t* partial, cudaStream_t st) {
    if (total <= 0) return cudaSuccess;
    if (vk_bits != 0 && vk_bits != 14) return cudaErrorNotSupported;
    auto kern = vk_bits == 14 ? k_aggv_partial_seg<14> : k_aggv_partial_seg<0>;
    int64_t blocks = (int64_t)persistent_grid(total, HWB, c.num_sms, resident_blocks(kern, RBS, 0));
    const int64_t ranges = seg_ranges(min(blocks, (int64_t)SEG_MAX_WARPS / HWB) * HWB);   // half-warps past the last range
    blocks = (ranges + HWB - 1) / HWB;                                                  // run dead trips only
    const int64_t per_hw = (total + ranges - 1) / ranges;
    if (per_hw > ((int64_t)1 << 20)) return cudaErrorInvalidValue;      // reduce64 bound (see the kernel)
    kern<<<(unsigned)blocks, RBS, 0, st>>>(c.m, c.scf, c.tab, static_cast<const uint16_t*>(vk_ntt), ch_pairs, ch_wt, ag_pairs,
                                           gid, total, n_agg, per_hw, partial);
    return cudaGetLastError();
}

cudaError_t launch_aggv_residues(const RingCtx& c, const int32_t* partial, int64_t nelem, uint16_t* out, cudaStream_t st) {
    if (nelem <= 0) return cudaSuccess;
    const int64_t need = (nelem + 255) / 256;
    k_aggv_residues<<<(unsigned)min(need, (int64_t)c.num_sms * 16), 256, 0, st>>>(c.m, partial, nelem, out);
    return cudaGetLastError();
}

cudaError_t launch_aggv_limits(const RingCtx& c, const int64_t* agg_off, int64_t n_agg, const int16_t* ag_sig, int64_t ag_cap,
                               uint8_t* verdict, cudaStream_t st) {
    if (n_agg <= 0) return cudaSuccess;
    const int64_t need = (n_agg + 255) / 256;
    k_aggv_limits<<<(unsigned)min(need, (int64_t)c.num_sms * 16), 256, 0, st>>>(agg_off, n_agg, ag_sig, (int64_t)c.l * D / 8,
                                                                                ag_cap, verdict);
    return cudaGetLastError();
}

cudaError_t launch_aggv_limits_packed(const RingCtx& c, const int64_t* agg_off, int64_t n_agg, const uint8_t* ag_packed, int bits,
                                      int bias, int64_t ag_cap, uint8_t* verdict, cudaStream_t st) {
    if (n_agg <= 0) return cudaSuccess;
    if (bits < 1 || bits > 16) return cudaErrorInvalidValue;
    const int64_t need = (n_agg + 255) / 256;
    k_aggv_limits_packed<<<(unsigned)min(need, (int64_t)c.num_sms * 16), 256, 0, st>>>(
        agg_off, n_agg, reinterpret_cast<const uint32_t*>(ag_packed), (int64_t)c.l * D, bits, (uint32_t)bias & 0xFFFFu, ag_cap,
        verdict);
    return cudaGetLastError();
}

}  // namespace lcb
