// Exact reuse of repeated blocks in the window pipeline (host_api.cu): group a window's cut blocks by their bytes, so
// that the nets run once per distinct block, and move results between compact (distinct) order and block order.
//
// A block's prediction depends on its cut net input alone (68x68 u8 luma, 3x34x34 u8 chroma), and a block's result
// does not depend on its position in a batch, so two byte-identical blocks get byte-identical maps, decode and flags.
//
// Grouping of n blocks (all on one stream, no host synchronisation):
//   pmp_block_hash_kernel    one warp per block: a 64-bit fingerprint (the sum over the block's 32-bit words w at word
//                            index k of splitmix64(k << 32 | w)), keeping the low hash_bits bits, and the identity index;
//   cub radix sort           (fingerprint, index) pairs on those bits; the sort is stable, so equal fingerprints keep
//                            ascending indices;
//   pmp_block_runs_kernel    + cub max-scan: for each sorted position, the first position of its fingerprint run;
//   pmp_block_match_kernel   one warp per sorted position p: compares block p byte for byte with the run's earlier
//                            blocks in order and stops at the first equal one.  Equal blocks have equal fingerprints and
//                            so share a run, in which indices ascend: the first equal block is the lowest equal index,
//                            rep[i].  A fingerprint collision costs compares, never a wrong rep;
//   cub exclusive sum        over rep[i] == i: the compact position of every distinct block;
//   pmp_block_slots_kernel   slot[i] (compact position of rep[i]), distinct[k] (block index of compact position k) and
//                            the distinct count.
// pmp_block_gather_kernel copies the distinct blocks into compact order; pmp_block_expand_kernel copies decoded maps,
// flags and the post-processed qt map from compact order back to block order.
#include "host.cuh"

#include <cub/cub.cuh>

namespace pmp {

namespace {

constexpr int BR_THREADS = 256, BR_WARPS = BR_THREADS / 32;

__device__ __forceinline__ unsigned long long mix64(unsigned long long x)
{
    x ^= x >> 30;
    x *= 0xbf58476d1ce4e5b9ull;
    x ^= x >> 27;
    x *= 0x94d049bb133111ebull;
    return x ^ (x >> 31);
}

// 16-byte words when every block starts 16-byte aligned, 4-byte words otherwise (chroma blocks are 3,468 bytes)
__device__ __forceinline__ bool vec16(const uint8_t *blocks, int block_bytes)
{
    return (block_bytes & 15) == 0 && (reinterpret_cast<uintptr_t>(blocks) & 15) == 0;
}

}  // namespace

// The kernels live outside the anonymous namespace, so that their names are stable in profiles.
__global__ void __launch_bounds__(BR_THREADS) pmp_block_hash_kernel(const uint8_t *__restrict__ blocks, int n,
                                                                    int block_bytes, int hash_bits,
                                                                    unsigned long long *__restrict__ keys,
                                                                    int *__restrict__ idx)
{
    const int b = blockIdx.x * BR_WARPS + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (b >= n) return;
    const uint8_t *p = blocks + (size_t)b * block_bytes;
    unsigned long long x = 0;
    if (vec16(blocks, block_bytes)) {
        const uint4 *q = reinterpret_cast<const uint4 *>(p);
        for (int k = lane; k < block_bytes / 16; k += 32) {
            const uint4 w = __ldg(q + k);
            const unsigned long long k4 = (unsigned long long)(4 * k) << 32;
            x += mix64(k4 | w.x) + mix64((k4 + (1ull << 32)) | w.y) + mix64((k4 + (2ull << 32)) | w.z) +
                 mix64((k4 + (3ull << 32)) | w.w);
        }
    } else {
        const uint32_t *q = reinterpret_cast<const uint32_t *>(p);
        for (int k = lane; k < block_bytes / 4; k += 32) x += mix64(((unsigned long long)k << 32) | __ldg(q + k));
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
    if (lane == 0) {
        keys[b] = hash_bits >= 64 ? x : x & ((1ull << hash_bits) - 1);
        idx[b] = b;
    }
}

__global__ void pmp_block_runs_kernel(const unsigned long long *__restrict__ keys, int n, int *__restrict__ head)
{
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p < n) head[p] = (p == 0 || keys[p] != keys[p - 1]) ? p : 0;
}

__device__ __forceinline__ bool warp_equal(const uint8_t *a, const uint8_t *b, int block_bytes, bool v16, int lane)
{
    if (v16) {
        const uint4 *x = reinterpret_cast<const uint4 *>(a), *y = reinterpret_cast<const uint4 *>(b);
        for (int k0 = 0; k0 < block_bytes / 16; k0 += 32) {
            const int k = k0 + lane;
            bool diff = false;
            if (k < block_bytes / 16) {
                const uint4 u = __ldg(x + k), v = __ldg(y + k);
                diff = u.x != v.x || u.y != v.y || u.z != v.z || u.w != v.w;
            }
            if (__any_sync(0xffffffffu, diff)) return false;
        }
    } else {
        const uint32_t *x = reinterpret_cast<const uint32_t *>(a), *y = reinterpret_cast<const uint32_t *>(b);
        for (int k0 = 0; k0 < block_bytes / 4; k0 += 32) {
            const int k = k0 + lane;
            const bool diff = k < block_bytes / 4 && __ldg(x + k) != __ldg(y + k);
            if (__any_sync(0xffffffffu, diff)) return false;
        }
    }
    return true;
}

__global__ void __launch_bounds__(BR_THREADS) pmp_block_match_kernel(const uint8_t *__restrict__ blocks, int n,
                                                                     int block_bytes, const int *__restrict__ sorted,
                                                                     const int *__restrict__ run_start,
                                                                     int *__restrict__ rep, int *__restrict__ is_rep)
{
    const int p = blockIdx.x * BR_WARPS + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (p >= n) return;
    const bool v16 = vec16(blocks, block_bytes);
    const int i = sorted[p];
    const uint8_t *bi = blocks + (size_t)i * block_bytes;
    int r = i;
    for (int q = run_start[p]; q < p; q++) {
        const int j = sorted[q];
        if (warp_equal(bi, blocks + (size_t)j * block_bytes, block_bytes, v16, lane)) {
            r = j;
            break;
        }
    }
    if (lane == 0) {
        rep[i] = r;
        is_rep[i] = r == i;
    }
}

__global__ void pmp_block_slots_kernel(const int *__restrict__ rep, const int *__restrict__ is_rep,
                                       const int *__restrict__ cslot, int n, int *__restrict__ slot,
                                       int *__restrict__ distinct, int *__restrict__ count)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    if (is_rep[i]) distinct[cslot[i]] = i;
    slot[i] = cslot[rep[i]];
    if (i == n - 1) *count = cslot[i] + is_rep[i];
}

__global__ void __launch_bounds__(BR_THREADS) pmp_block_gather_kernel(const uint8_t *__restrict__ blocks,
                                                                      const int *__restrict__ distinct, int nd,
                                                                      int block_bytes, uint8_t *__restrict__ out)
{
    const int k = blockIdx.x * BR_WARPS + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (k >= nd) return;
    const uint8_t *src = blocks + (size_t)distinct[k] * block_bytes;
    uint8_t *dst = out + (size_t)k * block_bytes;
    if (vec16(blocks, block_bytes) && (reinterpret_cast<uintptr_t>(out) & 15) == 0) {
        for (int w = lane; w < block_bytes / 16; w += 32)
            reinterpret_cast<uint4 *>(dst)[w] = __ldg(reinterpret_cast<const uint4 *>(src) + w);
    } else {
        for (int w = lane; w < block_bytes / 4; w += 32)
            reinterpret_cast<uint32_t *>(dst)[w] = __ldg(reinterpret_cast<const uint32_t *>(src) + w);
    }
}

// One warp per block i: hor [256] | ver [256] | dire [768] bytes (planes of `stride` blocks each), the u32 flags and,
// when src_qt is given, the 64-byte qt map, from compact position slot[i] to block position i.
__global__ void __launch_bounds__(BR_THREADS) pmp_block_expand_kernel(const int *__restrict__ slot, int n, long long stride,
                                                                      const uint8_t *__restrict__ src,
                                                                      uint8_t *__restrict__ dst,
                                                                      const uint32_t *__restrict__ src_flags,
                                                                      uint32_t *__restrict__ dst_flags,
                                                                      const uint8_t *__restrict__ src_qt,
                                                                      uint8_t *__restrict__ dst_qt)
{
    const int i = blockIdx.x * BR_WARPS + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (i >= n) return;
    const long long k = slot[i];
    const uint4 *s = reinterpret_cast<const uint4 *>(src);
    uint4 *d = reinterpret_cast<uint4 *>(dst);
    const long long hv = stride * 16;       // uint4 per hor (or ver) plane
    for (int w = lane; w < 80; w += 32) {
        const long long off = w < 16 ? 0 : w < 32 ? hv : 2 * hv;      // hor, ver, dire plane
        const int x = w < 16 ? w : w < 32 ? w - 16 : w - 32, per = w < 32 ? 16 : 48;
        d[off + (long long)i * per + x] = s[off + k * per + x];
    }
    if (src_qt && lane < 4)
        reinterpret_cast<uint4 *>(dst_qt)[(long long)i * 4 + lane] = reinterpret_cast<const uint4 *>(src_qt)[k * 4 + lane];
    if (lane == 0) dst_flags[i] = src_flags[k];
}

namespace {

struct MaxOp {
    __device__ __forceinline__ int operator()(int a, int b) const { return a > b ? a : b; }
};

size_t r256(size_t x) { return (x + 255) & ~(size_t)255; }

size_t cub_bytes(long long cap)
{
    size_t a = 0, b = 0, c = 0;
    cub::DoubleBuffer<unsigned long long> k(nullptr, nullptr);
    cub::DoubleBuffer<int> v(nullptr, nullptr);
    cub::DeviceRadixSort::SortPairs(nullptr, a, k, v, (int)cap, 0, 64);
    cub::DeviceScan::InclusiveScan(nullptr, b, (int *)nullptr, (int *)nullptr, MaxOp(), (int)cap);
    cub::DeviceScan::ExclusiveSum(nullptr, c, (int *)nullptr, (int *)nullptr, (int)cap);
    return r256(std::max(a, std::max(b, c)));
}

// The scratch of one grouping: fingerprints and indices (double-buffered for the sort), run starts, rep, rep flags,
// compact positions and cub's temporary storage.
struct Scratch {
    unsigned long long *keys[2];
    int *idx[2], *run, *rep, *is_rep, *cslot;
    void *temp;
    size_t temp_bytes;
};

Scratch scratch_of(char *buf, long long cap)
{
    Scratch s;
    const size_t w8 = r256((size_t)cap * 8), w4 = r256((size_t)cap * 4);
    s.keys[0] = (unsigned long long *)buf;
    s.keys[1] = (unsigned long long *)(buf + w8);
    char *p = buf + 2 * w8;
    int **ints[6] = {&s.idx[0], &s.idx[1], &s.run, &s.rep, &s.is_rep, &s.cslot};
    for (int **q : ints) {
        *q = (int *)p;
        p += w4;
    }
    s.temp = p;
    s.temp_bytes = cub_bytes(cap);
    return s;
}

size_t scratch_bytes(long long cap) { return 2 * r256((size_t)cap * 8) + 6 * r256((size_t)cap * 4) + cub_bytes(cap); }

unsigned grid_of(long long n, int per_cta) { return (unsigned)((n + per_cta - 1) / per_cta); }

}  // namespace

size_t group_bytes(long long cap)
{
    return scratch_bytes(cap) + GROUP_SLOTS * 2 * 2 * r256((size_t)cap * 4) + 256;
}

Groups groups_of(char *buf, long long cap, int slot, int comp)
{
    const size_t w4 = r256((size_t)cap * 4);
    char *p = buf + scratch_bytes(cap) + (size_t)(2 * slot + comp) * 2 * w4;
    Groups g;
    g.slot = (int *)p;
    g.distinct = (int *)(p + w4);
    g.count = (int *)(buf + scratch_bytes(cap) + GROUP_SLOTS * 2 * 2 * w4) + 2 * slot + comp;
    return g;
}

int group_blocks(Handle *h, char *buf, long long cap, const uint8_t *blocks, int n, int block_bytes, int hash_bits,
                 int *rep_out, const Groups &g, cudaStream_t st)
{
    if (n <= 0) return PMP_OK;
    if (n > cap) {
        set_error("internal: %d blocks to group, scratch for %lld", n, cap);
        return PMP_ERR_STATE;
    }
    Scratch s = scratch_of(buf, cap);
    int *rep = rep_out ? rep_out : s.rep;
    pmp_block_hash_kernel<<<grid_of(n, BR_WARPS), BR_THREADS, 0, st>>>(blocks, n, block_bytes, hash_bits, s.keys[0],
                                                                       s.idx[0]);
    h->launches++;
    PMP_CUDA(cudaGetLastError());
    cub::DoubleBuffer<unsigned long long> keys(s.keys[0], s.keys[1]);
    cub::DoubleBuffer<int> idx(s.idx[0], s.idx[1]);
    if (hash_bits > 0) {        // with 0 bits every key is 0: the identity order is already sorted
        size_t need = 0;
        cub::DeviceRadixSort::SortPairs(nullptr, need, keys, idx, n, 0, hash_bits, st);
        if (need > s.temp_bytes) {
            set_error("internal: the radix sort of %d blocks needs %zu bytes, the scratch holds %zu", n, need, s.temp_bytes);
            return PMP_ERR_STATE;
        }
        PMP_CUDA(cub::DeviceRadixSort::SortPairs(s.temp, need, keys, idx, n, 0, hash_bits, st));
    }
    pmp_block_runs_kernel<<<grid_of(n, 256), 256, 0, st>>>(keys.Current(), n, s.cslot);
    h->launches++;
    PMP_CUDA(cudaGetLastError());
    size_t need = s.temp_bytes;
    PMP_CUDA(cub::DeviceScan::InclusiveScan(s.temp, need, s.cslot, s.run, MaxOp(), n, st));
    pmp_block_match_kernel<<<grid_of(n, BR_WARPS), BR_THREADS, 0, st>>>(blocks, n, block_bytes, idx.Current(), s.run, rep,
                                                                        s.is_rep);
    h->launches++;
    PMP_CUDA(cudaGetLastError());
    need = s.temp_bytes;
    PMP_CUDA(cub::DeviceScan::ExclusiveSum(s.temp, need, s.is_rep, s.cslot, n, st));
    pmp_block_slots_kernel<<<grid_of(n, 256), 256, 0, st>>>(rep, s.is_rep, s.cslot, n, g.slot, g.distinct, g.count);
    h->launches++;
    PMP_CUDA(cudaGetLastError());
    return PMP_OK;
}

int gather_blocks(Handle *h, const uint8_t *blocks, const int *distinct, int nd, int block_bytes, uint8_t *out,
                  cudaStream_t st)
{
    if (nd <= 0) return PMP_OK;
    pmp_block_gather_kernel<<<grid_of(nd, BR_WARPS), BR_THREADS, 0, st>>>(blocks, distinct, nd, block_bytes, out);
    h->launches++;
    PMP_CUDA(cudaGetLastError());
    return PMP_OK;
}

int expand_blocks(Handle *h, const int *slot, int n, long long stride, const uint8_t *src, uint8_t *dst,
                  const uint32_t *src_flags, uint32_t *dst_flags, const uint8_t *src_qt, uint8_t *dst_qt, cudaStream_t st)
{
    if (n <= 0) return PMP_OK;
    pmp_block_expand_kernel<<<grid_of(n, BR_WARPS), BR_THREADS, 0, st>>>(slot, n, stride, src, dst, src_flags, dst_flags,
                                                                         src_qt, dst_qt);
    h->launches++;
    PMP_CUDA(cudaGetLastError());
    return PMP_OK;
}

}  // namespace pmp
