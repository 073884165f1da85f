// order.cu — the per-group sort of content strings and the gathers that put a content-mode BKLM batch into sorted order
// on the device (sm_100a).
//
// BKLM hashes and sums the items of an aggregate sorted by str(otvk) (prepare_make_agg_coefs, a stable sort).  In
// content mode those strings are the 57-byte rows of lcb_content_str_batch, so the order is a stable per-group sort of
// 57-byte rows in unsigned byte order.  A row is held as eight big-endian 64-bit words (bytes 57..63 zero), whose
// lexicographic order is memcmp order; ties are broken by the item index, which makes every path stable.
//   k_content_order        groups of at most small_max items: one thread per item, rank = the number of rows of its
//                          group that are smaller, or equal with a lower index (the shipped ag_cap = 2 case);
//   k_content_order_block  groups of at most block_max (<= ORDER_BLOCK_MAX) items: one block per group, a bitonic sort
//                          of item indices over the rows staged in shared memory;
//   larger groups          all of them at once: a stable LSD radix sort (CUB) over the eight words, then over the group.
//   k_gather_rows          dst[k] = src[index[k]], one warp per row, 16-, 4- or 1-byte units;
//   k_ragged_*             the exclusive scan of the gathered lengths (two-level: tile scans, then one block over the tile
//                          sums), then one warp per item copies the bytes.
// An index outside [0, n_src) gives an all-zero row or an empty item: no kernel reads outside its source buffer.
#include <cub/device/device_radix_sort.cuh>

#include "engine.h"

namespace lcb {

namespace {

constexpr int ROW = 57;
constexpr int OBS = 512;                 // threads of k_content_order_block
constexpr int TILE_THREADS = 256;        // k_ragged_scan_tiles: 4 items per thread
constexpr int TILE = 4 * TILE_THREADS;

__device__ __forceinline__ uint64_t row_word(const uint8_t* __restrict__ p, int k) {
    uint64_t v = 0;
#pragma unroll
    for (int b = 0; b < 8; ++b) {
        const int at = 8 * k + b;
        v = (v << 8) | (at < ROW ? (uint64_t)__ldg(p + at) : 0ull);
    }
    return v;
}

__device__ __forceinline__ void row_words(const uint8_t* __restrict__ p, uint64_t (&w)[8]) {
#pragma unroll
    for (int k = 0; k < 8; ++k) w[k] = row_word(p, k);
}

// (a, ia) < (b, ib): row a before row b, equal rows by index
__device__ __forceinline__ bool before(const uint64_t (&a)[8], int64_t ia, const uint64_t (&b)[8], int64_t ib) {
#pragma unroll
    for (int k = 0; k < 8; ++k)
        if (a[k] != b[k]) return a[k] < b[k];
    return ia < ib;
}

__global__ void __launch_bounds__(256) k_content_order(const int64_t* __restrict__ agg_off, const int32_t* __restrict__ gid,
                                                       int64_t n_agg, int64_t total, const uint8_t* __restrict__ rows,
                                                       int small_max, int64_t* __restrict__ order) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int g = __ldg(gid + i);
        LCB_CHECK(g >= 0 && g < n_agg);
        const int64_t a0 = __ldg(agg_off + g), a1 = __ldg(agg_off + g + 1);
        LCB_CHECK(a0 >= 0 && a0 <= i && i < a1 && a1 <= total);
        if (a1 - a0 > small_max) continue;
        uint64_t mine[8], other[8];
        row_words(rows + i * ROW, mine);
        int64_t rank = 0;
        for (int64_t j = a0; j < a1; ++j) {
            if (j == i) continue;
            row_words(rows + j * ROW, other);
            rank += before(other, j, mine, i) ? 1 : 0;
        }
        LCB_CHECK(a0 + rank < a1);
        order[a0 + rank] = i;
    }
}

// Keys in shared memory as [8][ORDER_BLOCK_MAX] words, then int32 idx[ORDER_BLOCK_MAX]; slots cnt .. P-1 of the padded
// power of two P sort last.
__device__ __forceinline__ bool after_sm(const uint64_t* __restrict__ keys, int x, int y, int cnt) {
    if (x >= cnt || y >= cnt) return x >= cnt && (y < cnt || x > y);
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        const uint64_t a = keys[k * ORDER_BLOCK_MAX + x], b = keys[k * ORDER_BLOCK_MAX + y];
        if (a != b) return a > b;
    }
    return x > y;
}

__global__ void __launch_bounds__(OBS) k_content_order_block(const int64_t* __restrict__ agg_off, const int32_t* __restrict__ groups,
                                                             int64_t n_agg, int64_t total, const uint8_t* __restrict__ rows,
                                                             int64_t* __restrict__ order) {
    extern __shared__ uint64_t keys[];
    int32_t* idx = reinterpret_cast<int32_t*>(keys + 8 * ORDER_BLOCK_MAX);
    const int g = __ldg(groups + blockIdx.x);
    LCB_CHECK(g >= 0 && g < n_agg);
    const int64_t a0 = __ldg(agg_off + g), a1 = __ldg(agg_off + g + 1);
    LCB_CHECK(a0 >= 0 && a0 <= a1 && a1 <= total && a1 - a0 <= ORDER_BLOCK_MAX);
    const int cnt = (int)(a1 - a0);
    int P = 1;
    while (P < cnt) P <<= 1;
    for (int t = threadIdx.x; t < 8 * ORDER_BLOCK_MAX; t += OBS) keys[t] = 0;
    __syncthreads();
    // byte k of the group's rows: item k / 57, position k % 57 -> word pos / 8, big-endian byte (pos % 8) of it
    uint8_t* kb = reinterpret_cast<uint8_t*>(keys);
    const uint8_t* src = rows + a0 * ROW;
    for (int k = threadIdx.x; k < cnt * ROW; k += OBS) {
        LCB_CHECK(a0 * ROW + k < total * ROW);
        const int item = k / ROW, pos = k - item * ROW;
        kb[((pos >> 3) * ORDER_BLOCK_MAX + item) * 8 + (7 - (pos & 7))] = __ldg(src + k);
    }
    for (int t = threadIdx.x; t < P; t += OBS) idx[t] = t;
    for (int k = 2; k <= P; k <<= 1) {
        for (int j = k >> 1; j > 0; j >>= 1) {
            __syncthreads();
            for (int t = threadIdx.x; t < P; t += OBS) {
                const int u = t ^ j;
                if (u <= t) continue;
                const int x = idx[t], y = idx[u];
                const bool up = (t & k) == 0;
                if (up ? after_sm(keys, x, y, cnt) : after_sm(keys, y, x, cnt)) {
                    idx[t] = y;
                    idx[u] = x;
                }
            }
        }
    }
    __syncthreads();
    for (int t = threadIdx.x; t < cnt; t += OBS) order[a0 + t] = a0 + idx[t];
}

// ---- the largest groups: m items of L groups, group k = items a0[k] .. a0[k] + (base[k+1] - base[k]), at positions
// base[k] .. base[k+1] of the concatenation
__device__ __forceinline__ int group_of(const int64_t* __restrict__ v, int L, int64_t x) {
    int lo = 0, hi = L - 1;                                   // the last k with v[k] <= x
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (__ldg(v + mid) <= x) lo = mid;
        else hi = mid - 1;
    }
    return lo;
}

__global__ void __launch_bounds__(256) k_order_large_init(const int64_t* __restrict__ a0, const int64_t* __restrict__ base, int L,
                                                          int64_t m, int32_t* __restrict__ perm) {
    for (int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; p < m; p += (int64_t)gridDim.x * blockDim.x) {
        const int k = group_of(base, L, p);
        perm[p] = (int32_t)(__ldg(a0 + k) + (p - __ldg(base + k)));
    }
}

// word w of the row of item perm[p]; w = 8: the group of perm[p]
__global__ void __launch_bounds__(256) k_order_large_keys(const uint8_t* __restrict__ rows, int64_t total, const int32_t* __restrict__ perm,
                                                          int64_t m, int w, const int64_t* __restrict__ a0, int L,
                                                          uint64_t* __restrict__ keys) {
    for (int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; p < m; p += (int64_t)gridDim.x * blockDim.x) {
        const int64_t i = __ldg(perm + p);
        LCB_CHECK(i >= 0 && i < total);
        keys[p] = w < 8 ? row_word(rows + i * ROW, w) : (uint64_t)group_of(a0, L, i);
    }
}

__global__ void __launch_bounds__(256) k_order_large_scatter(const int32_t* __restrict__ perm, int64_t m, const int64_t* __restrict__ a0,
                                                             const int64_t* __restrict__ base, int L, int64_t total,
                                                             int64_t* __restrict__ order) {
    for (int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; p < m; p += (int64_t)gridDim.x * blockDim.x) {
        const int k = group_of(base, L, p);
        const int64_t at = __ldg(a0 + k) + (p - __ldg(base + k));
        LCB_CHECK(at >= 0 && at < total);
        order[at] = __ldg(perm + p);
    }
}

// ---- gathers
template <typename U>
__global__ void __launch_bounds__(256) k_gather_rows(const U* __restrict__ src, int64_t n_src, int64_t units,
                                                     const int64_t* __restrict__ index, int64_t n, U* __restrict__ dst) {
    const int lane = threadIdx.x & 31;
    for (int64_t k = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; k < n; k += ((int64_t)gridDim.x * blockDim.x) >> 5) {
        const int64_t s = __ldg(index + k);
        const bool ok = s >= 0 && s < n_src;
        const U* from = src + (ok ? s : 0) * units;
        U* to = dst + k * units;
#pragma unroll 4
        for (int64_t u = lane; u < units; u += 32) {
            LCB_CHECK(!ok || s * units + u < n_src * units);
            to[u] = ok ? from[u] : U{};
        }
    }
}

__device__ __forceinline__ int64_t item_len(const int64_t* __restrict__ off, int64_t n_src, const int64_t* __restrict__ index,
                                            int64_t n, int64_t k) {
    if (k >= n) return 0;
    const int64_t s = __ldg(index + k);
    if (s < 0 || s >= n_src) return 0;
    const int64_t len = __ldg(off + s + 1) - __ldg(off + s);
    return len > 0 ? len : 0;
}

// exclusive scan of v over the block; *sum = the block total
template <int THREADS>
__device__ __forceinline__ int64_t block_scan(int64_t v, int64_t* __restrict__ warp_sums, int64_t* sum) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    int64_t x = v;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const int64_t y = __shfl_up_sync(0xffffffffu, x, d);
        if (lane >= d) x += y;
    }
    if (lane == 31) warp_sums[wid] = x;
    __syncthreads();
    if (wid == 0) {
        int64_t s = lane < THREADS / 32 ? warp_sums[lane] : 0;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const int64_t y = __shfl_up_sync(0xffffffffu, s, d);
            if (lane >= d) s += y;
        }
        if (lane < THREADS / 32) warp_sums[lane] = s;          // inclusive over warps
    }
    __syncthreads();
    const int64_t before = (wid > 0 ? warp_sums[wid - 1] : 0) + x - v;
    *sum = warp_sums[THREADS / 32 - 1];
    __syncthreads();                                          // warp_sums is reused by the next call
    return before;
}

// out_off[k + 1] = the gathered bytes of items tile_start .. k (inclusive, within the tile); tile_sum[t] = the tile total
__global__ void __launch_bounds__(TILE_THREADS) k_ragged_scan_tiles(const int64_t* __restrict__ off, int64_t n_src,
                                                                    const int64_t* __restrict__ index, int64_t n,
                                                                    int64_t* __restrict__ out_off, int64_t* __restrict__ tile_sum) {
    __shared__ int64_t ws[32];
    const int64_t k0 = (int64_t)blockIdx.x * TILE + 4 * threadIdx.x;
    int64_t len[4], mine = 0;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        len[j] = item_len(off, n_src, index, n, k0 + j);
        mine += len[j];
    }
    int64_t sum;
    int64_t run = block_scan<TILE_THREADS>(mine, ws, &sum);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        run += len[j];
        if (k0 + j < n) out_off[k0 + j + 1] = run;
    }
    if (threadIdx.x == 0) tile_sum[blockIdx.x] = sum;
}

// tile_sum[0 .. ntiles) -> exclusive prefix in place, tile_sum[ntiles] = total; one block
__global__ void __launch_bounds__(1024) k_ragged_scan_carry(int64_t* __restrict__ tile_sum, int64_t ntiles) {
    __shared__ int64_t ws[32];
    int64_t carry = 0;
    for (int64_t b = 0; b < ntiles; b += 1024) {
        const int64_t t = b + threadIdx.x;
        const int64_t v = t < ntiles ? tile_sum[t] : 0;
        int64_t sum;
        const int64_t ex = block_scan<1024>(v, ws, &sum);
        if (t < ntiles) tile_sum[t] = carry + ex;
        carry += sum;
    }
    if (threadIdx.x == 0) tile_sum[ntiles] = carry;
}

__global__ void __launch_bounds__(256) k_ragged_scan_add(const int64_t* __restrict__ tile_base, int64_t n, int64_t* __restrict__ out_off) {
    for (int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; k < n; k += (int64_t)gridDim.x * blockDim.x)
        out_off[k + 1] += __ldg(tile_base + k / TILE);
    if (blockIdx.x == 0 && threadIdx.x == 0) out_off[0] = 0;
}

// item k -> out[out_off[k] ..): blob[off[index[k]] - shift .. off[index[k] + 1] - shift); nothing past out_cap is written
__global__ void __launch_bounds__(256) k_gather_ragged(const uint8_t* __restrict__ blob, int64_t shift, const int64_t* __restrict__ off,
                                                       int64_t n_src, const int64_t* __restrict__ index, int64_t n,
                                                       const int64_t* __restrict__ out_off, int64_t out_cap,
                                                       uint8_t* __restrict__ out) {
    const int lane = threadIdx.x & 31;
    for (int64_t k = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; k < n; k += ((int64_t)gridDim.x * blockDim.x) >> 5) {
        const int64_t s = __ldg(index + k);
        if (s < 0 || s >= n_src) continue;
        const int64_t b0 = __ldg(off + s), len = __ldg(off + s + 1) - b0, o0 = __ldg(out_off + k);
        LCB_CHECK(len <= 0 || (b0 - shift >= 0 && o0 >= 0 && o0 + len <= out_cap));
        if (len <= 0 || o0 < 0 || o0 + len > out_cap) continue;
        const uint8_t* from = blob + (b0 - shift);
        uint8_t* to = out + o0;
        for (int64_t t = lane; t < len; t += 32) to[t] = __ldg(from + t);
    }
}

unsigned grid_for(int64_t items, int per_block, int num_sms) {
    const int64_t blocks = (items + per_block - 1) / per_block;
    const int64_t cap = (int64_t)num_sms * 16;
    return (unsigned)(blocks < 1 ? 1 : (blocks < cap ? blocks : cap));
}

}  // namespace

cudaError_t launch_content_order_small(const int64_t* agg_off, const int32_t* gid, int64_t n_agg, int64_t total,
                                       const uint8_t* rows, int small_max, int64_t* order, int num_sms, cudaStream_t st) {
    if (total <= 0 || small_max < 1) return cudaSuccess;
    k_content_order<<<grid_for(total, 256, num_sms), 256, 0, st>>>(agg_off, gid, n_agg, total, rows, small_max, order);
    return cudaGetLastError();
}

cudaError_t launch_content_order_block(const int64_t* agg_off, const int32_t* groups, int64_t n_groups, int64_t n_agg,
                                       int64_t total, const uint8_t* rows, int64_t* order, cudaStream_t st) {
    if (n_groups <= 0) return cudaSuccess;
    const size_t smem = (size_t)ORDER_BLOCK_MAX * (8 * sizeof(uint64_t) + sizeof(int32_t));
    cudaError_t e = cudaFuncSetAttribute(k_content_order_block, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    for (int64_t first = 0; first < n_groups; first += (int64_t)1 << 30) {    // grid.x limit is 2^31 - 1
        const int64_t cnt = n_groups - first < ((int64_t)1 << 30) ? n_groups - first : ((int64_t)1 << 30);
        k_content_order_block<<<(unsigned)cnt, OBS, smem, st>>>(agg_off, groups + first, n_agg, total, rows, order);
        if ((e = cudaGetLastError()) != cudaSuccess) return e;
    }
    return cudaSuccess;
}

cudaError_t content_order_large_scratch(int64_t m, size_t* bytes) {
    size_t temp = 0;
    cudaError_t e = cub::DeviceRadixSort::SortPairs(nullptr, temp, static_cast<const uint64_t*>(nullptr),
                                                    static_cast<uint64_t*>(nullptr), static_cast<const int32_t*>(nullptr),
                                                    static_cast<int32_t*>(nullptr), (int)m);
    *bytes = temp;
    return e;
}

cudaError_t launch_content_order_large(const uint8_t* rows, int64_t total, const int64_t* a0, const int64_t* base, int L, int64_t m,
                                       uint64_t* keys, int32_t* perm, void* temp, size_t temp_bytes, int64_t* order,
                                       int num_sms, cudaStream_t st) {
    if (m <= 0) return cudaSuccess;
    // keys / perm hold two buffers of m each
    cub::DoubleBuffer<uint64_t> kb(keys, keys + m);
    cub::DoubleBuffer<int32_t> vb(perm, perm + m);
    const unsigned grid = grid_for(m, 256, num_sms);
    k_order_large_init<<<grid, 256, 0, st>>>(a0, base, L, m, vb.Current());
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    int gbits = 0;
    while ((1 << gbits) < L) ++gbits;
    // least significant first: word 7 (one byte, bits 56..63), words 6 .. 0, then the group
    for (int w = 7; w >= -1; --w) {
        const int key = w < 0 ? 8 : w;
        if (key == 8 && gbits == 0) break;
        k_order_large_keys<<<grid, 256, 0, st>>>(rows, total, vb.Current(), m, key, a0, L, kb.Current());
        if ((e = cudaGetLastError()) != cudaSuccess) return e;
        const int lo = key == 7 ? 56 : 0, hi = key == 8 ? gbits : 64;
        size_t tb = temp_bytes;
        if ((e = cub::DeviceRadixSort::SortPairs(temp, tb, kb, vb, (int)m, lo, hi, st)) != cudaSuccess) return e;
    }
    k_order_large_scatter<<<grid, 256, 0, st>>>(vb.Current(), m, a0, base, L, total, order);
    return cudaGetLastError();
}

cudaError_t launch_gather_rows(const uint8_t* src, int64_t n_src, int64_t row_bytes, const int64_t* index, int64_t n, uint8_t* dst,
                               int num_sms, cudaStream_t st) {
    if (n <= 0) return cudaSuccess;
    const unsigned grid = grid_for(n, 8, num_sms);       // one row per warp, 8 warps per block
    const uintptr_t a = reinterpret_cast<uintptr_t>(src) | reinterpret_cast<uintptr_t>(dst);
    if (row_bytes % 16 == 0 && a % 16 == 0)
        k_gather_rows<uint4><<<grid, 256, 0, st>>>(reinterpret_cast<const uint4*>(src), n_src, row_bytes / 16, index, n,
                                                   reinterpret_cast<uint4*>(dst));
    else if (row_bytes % 4 == 0 && a % 4 == 0)
        k_gather_rows<uint32_t><<<grid, 256, 0, st>>>(reinterpret_cast<const uint32_t*>(src), n_src, row_bytes / 4, index, n,
                                                      reinterpret_cast<uint32_t*>(dst));
    else
        k_gather_rows<uint8_t><<<grid, 256, 0, st>>>(src, n_src, row_bytes, index, n, dst);
    return cudaGetLastError();
}

int64_t ragged_scan_tiles(int64_t n) { return (n + TILE - 1) / TILE; }

cudaError_t launch_ragged_scan(const int64_t* off, int64_t n_src, const int64_t* index, int64_t n, int64_t* tile_sum,
                               int64_t* out_off, int num_sms, cudaStream_t st) {
    if (n <= 0) return cudaSuccess;
    const int64_t ntiles = ragged_scan_tiles(n);
    if (ntiles >= ((int64_t)1 << 31)) return cudaErrorInvalidValue;
    k_ragged_scan_tiles<<<(unsigned)ntiles, TILE_THREADS, 0, st>>>(off, n_src, index, n, out_off, tile_sum);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    k_ragged_scan_carry<<<1, 1024, 0, st>>>(tile_sum, ntiles);
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
    k_ragged_scan_add<<<grid_for(n, 256, num_sms), 256, 0, st>>>(tile_sum, n, out_off);
    return cudaGetLastError();
}

cudaError_t launch_gather_ragged(const uint8_t* blob, int64_t shift, const int64_t* off, int64_t n_src, const int64_t* index,
                                 int64_t n, const int64_t* out_off, int64_t out_cap, uint8_t* out, int num_sms, cudaStream_t st) {
    if (n <= 0) return cudaSuccess;
    k_gather_ragged<<<grid_for(n, 8, num_sms), 256, 0, st>>>(blob, shift, off, n_src, index, n, out_off, out_cap, out);
    return cudaGetLastError();
}

}  // namespace lcb
