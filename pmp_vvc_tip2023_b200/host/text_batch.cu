// pmp_format_texts: the PartitionMat text body (Map2Partition.py:405-412, one decimal integer and '\n' per value) of up
// to TEXTS_MAX int8 vectors in one launch, without a host synchronisation.
//
// Single-pass scan with decoupled look-back (Merrill & Garland, "Single-pass Parallel Prefix Scan with Decoupled
// Look-back", 2016): every CTA formats one tile of one vector.  It counts its tile's bytes (2 per value, 3 for -1),
// publishes that aggregate in its tile status word, then walks back over the same vector's earlier tiles until it finds
// an inclusive prefix, publishes its own, formats the tile into shared memory at the destination's 16-byte phase and
// stores it with 16-byte stores.  Tiles of a vector are consecutive CTAs, so a CTA only ever waits on lower-numbered
// ones.  A status word is (epoch << 34) | (flag << 32) | bytes: the epoch changes with every launch, so the words need
// no clearing between launches.
#include "host.cuh"

#include <map>
#include <mutex>

namespace pmp {

constexpr int TT_THREADS = 256, TT_PER_THREAD = 16, TT_TILE = TT_THREADS * TT_PER_THREAD;
constexpr unsigned long long ST_AGGREGATE = 1ull << 32, ST_PREFIX = 2ull << 32, ST_FLAGS = 3ull << 32;
constexpr int EPOCH_SHIFT = 34;
constexpr unsigned EPOCH_LIMIT = 1u << 30;

struct TextBatch {
    const int8_t *values[TEXTS_MAX];
    char *text[TEXTS_MAX];
    long long n[TEXTS_MAX];
    int tile0[TEXTS_MAX + 1];       // first tile (CTA) of each vector; tile0[m] = number of tiles
    int m;
    int64_t *n_bytes;
    unsigned long long *status;     // one word per tile
    unsigned long long epoch;       // already shifted by EPOCH_SHIFT
};

__device__ __forceinline__ unsigned long long ld_status(const unsigned long long *p)
{
    unsigned long long v;
    asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}

__device__ __forceinline__ void st_status(unsigned long long *p, unsigned long long v)
{
    asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}

__global__ void __launch_bounds__(TT_THREADS) pmp_format_texts_kernel(const TextBatch b)
{
    __shared__ __align__(16) char stage[3 * TT_TILE + 16];
    __shared__ int warp_sum[TT_THREADS / 32];
    __shared__ unsigned long long s_prefix;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (blockIdx.x == 0 && tid < b.m && b.n[tid] == 0) b.n_bytes[tid] = 0;
    if ((int)blockIdx.x >= b.tile0[b.m]) return;        // the one CTA of a launch whose vectors are all empty
    int vi = 0;
    while ((int)blockIdx.x >= b.tile0[vi + 1]) vi++;
    const int t = blockIdx.x - b.tile0[vi], last = b.tile0[vi + 1] - b.tile0[vi] - 1;
    const long long n = b.n[vi], i0 = (long long)t * TT_TILE + (long long)tid * TT_PER_THREAD;
    const int8_t *src = b.values[vi] + i0;

    // this thread's 16 consecutive values: one 16-byte load where the tile is full and aligned
    int8_t v[TT_PER_THREAD];
    const int cnt = (int)max(0LL, min((long long)TT_PER_THREAD, n - i0));
    if (cnt == TT_PER_THREAD && (reinterpret_cast<uintptr_t>(src) & 15) == 0) {
        const int4 q = __ldg(reinterpret_cast<const int4 *>(src));
        memcpy(v, &q, 16);
    } else {
#pragma unroll
        for (int k = 0; k < TT_PER_THREAD; k++) v[k] = k < cnt ? src[k] : 0;
    }
    int mine = 0;
#pragma unroll
    for (int k = 0; k < TT_PER_THREAD; k++) mine += k < cnt ? 2 + (v[k] < 0) : 0;

    // block-wide exclusive scan of the per-thread byte counts
    int incl = mine;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int x = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += x;
    }
    if (lane == 31) warp_sum[warp] = incl;
    __syncthreads();
    int off = incl - mine, total = 0;
#pragma unroll
    for (int w = 0; w < TT_THREADS / 32; w++) {
        off += w < warp ? warp_sum[w] : 0;
        total += warp_sum[w];
    }

    // decoupled look-back over this vector's earlier tiles
    if (tid == 0) {
        unsigned long long *st = b.status + blockIdx.x;
        unsigned long long prefix = 0;
        if (t > 0) {
            st_status(st, b.epoch | ST_AGGREGATE | (unsigned)total);
            for (int j = (int)blockIdx.x - 1;; j--) {
                unsigned long long w;
                do {
                    w = ld_status(b.status + j);
                } while ((w >> EPOCH_SHIFT) != (b.epoch >> EPOCH_SHIFT) || (w & ST_FLAGS) == 0);
                prefix += (unsigned)w;
                if ((w & ST_FLAGS) == ST_PREFIX) break;
            }
        }
        st_status(st, b.epoch | ST_PREFIX | (unsigned)(prefix + total));
        if (t == last) b.n_bytes[vi] = (int64_t)(prefix + total);
        s_prefix = prefix;
    }
    __syncthreads();

    // format at the destination's 16-byte phase, then store whole aligned 16-byte chunks
    char *dst = b.text[vi] + s_prefix;
    const int lead = (int)(reinterpret_cast<uintptr_t>(dst) & 15), end = lead + total;
    char *p = stage + lead + off;
#pragma unroll
    for (int k = 0; k < TT_PER_THREAD; k++) {
        if (k < cnt) {
            int x = v[k];
            if (x < 0) { *p++ = '-'; x = -x; }
            *p++ = (char)('0' + x);
            *p++ = '\n';
        }
    }
    __syncthreads();
    char *abase = dst - lead;
    for (int c = tid; c < (end + 15) / 16; c += TT_THREADS) {
        const int b0 = 16 * c;
        if (b0 >= lead && b0 + 16 <= end) {
            *reinterpret_cast<int4 *>(abase + b0) = *reinterpret_cast<const int4 *>(stage + b0);
        } else {
            for (int k = max(b0, lead); k < min(b0 + 16, end); k++) abase[k] = stage[k];
        }
    }
}

namespace {

struct TextStatus {
    unsigned long long *words = nullptr;
    long long cap = 0;
    unsigned epoch = 0;
};

std::mutex g_text_mu;
std::map<const Handle *, TextStatus> g_text;     // a handle is used by one thread at a time; the map by all

TextStatus &text_status_of(const Handle *h)
{
    std::lock_guard<std::mutex> lock(g_text_mu);
    return g_text[h];
}

long long tiles_of(long long n) { return (n + TT_TILE - 1) / TT_TILE; }

// Zeroed words for at least `tiles` tiles.  Growing or clearing waits for every launch that may still read the old words.
int ensure_words(TextStatus &ts, long long tiles)
{
    if (tiles <= ts.cap && ts.words) return PMP_OK;
    PMP_CUDA(cudaDeviceSynchronize());
    if (ts.words) PMP_CUDA(cudaFree(ts.words));
    ts.words = nullptr;
    ts.cap = 0;
    const long long cap = std::max(tiles, 1024LL);
    PMP_CUDA(cudaMalloc((void **)&ts.words, (size_t)cap * 8));
    PMP_CUDA(cudaMemset(ts.words, 0, (size_t)cap * 8));
    PMP_CUDA(cudaDeviceSynchronize());
    ts.cap = cap;
    ts.epoch = 0;
    return PMP_OK;
}

}  // namespace

int reserve_text_status(Handle *h, int m, long long n)
{
    return ensure_words(text_status_of(h), (long long)m * tiles_of(n));
}

int format_texts(Handle *h, int m, const int8_t *const *values, const int64_t *n, char *const *text, int64_t *n_bytes,
                 cudaStream_t s)
{
    TextBatch b{};
    b.m = m;
    b.n_bytes = n_bytes;
    long long tiles = 0;
    for (int i = 0; i < m; i++) {
        b.values[i] = values[i];
        b.text[i] = text[i];
        b.n[i] = n[i];
        b.tile0[i] = (int)tiles;
        tiles += tiles_of(n[i]);
    }
    b.tile0[m] = (int)tiles;
    TextStatus &ts = text_status_of(h);
    int rc = ensure_words(ts, tiles);
    if (rc) return rc;
    if (++ts.epoch == EPOCH_LIMIT) {            // the epoch field wraps: clear the words once, start again at 1
        PMP_CUDA(cudaDeviceSynchronize());
        PMP_CUDA(cudaMemset(ts.words, 0, (size_t)ts.cap * 8));
        PMP_CUDA(cudaDeviceSynchronize());
        ts.epoch = 1;
    }
    b.status = ts.words;
    b.epoch = (unsigned long long)ts.epoch << EPOCH_SHIFT;
    pmp_format_texts_kernel<<<(unsigned)std::max(tiles, 1LL), TT_THREADS, 0, s>>>(b);
    h->launches++;
    PMP_CUDA(cudaGetLastError());
    return PMP_OK;
}

void release_text_status(const Handle *h)
{
    TextStatus ts;
    {
        std::lock_guard<std::mutex> lock(g_text_mu);
        auto it = g_text.find(h);
        if (it == g_text.end()) return;
        ts = it->second;
        g_text.erase(it);
    }
    if (ts.words) {
        cudaSetDevice(h->device);
        cudaDeviceSynchronize();
        cudaFree(ts.words);
    }
}

}  // namespace pmp
