// Internal interface between the host-level sources (host_api.cu, text_batch.cu).
#pragma once
#include "../csrc/handle.cuh"

namespace pmp {

constexpr int TEXTS_MAX = 8;                          // vectors per pmp_format_texts launch
constexpr long long TEXT_MAX_VALUES = 1LL << 30;      // per vector: its text offsets fit the 32-bit tile status values

// pmp_format_texts without the argument checks of the public entry point (text_batch.cu).  Asynchronous on `s`; the
// per-tile status words are the handle's, so launches of one handle must not run concurrently on different streams.
int format_texts(Handle *h, int m, const int8_t *const *values, const int64_t *n, char *const *text, int64_t *n_bytes,
                 cudaStream_t s);
// Grows the handle's tile status words to hold `m` vectors of `n` values each, so that later format_texts calls of at
// most that size do not allocate (an allocation synchronises the device).
int reserve_text_status(Handle *h, int m, long long n);
// Frees the tile status words (pmp_destroy).
void release_text_status(const Handle *h);

// ---- block_reuse.cu: grouping of byte-identical blocks --------------------------------------------------------------
constexpr int GROUP_SLOTS = 2;        // window slots of the pipeline, each with the groups of both components
// One grouping's results (device): slot[i] = compact position of block i's lowest equal block, distinct[k] = block
// index of compact position k (ascending), *count = number of distinct blocks.
struct Groups { int *slot, *distinct, *count; };
// Bytes of a grouping buffer for up to `cap` blocks: one grouping's scratch plus the Groups of GROUP_SLOTS x 2 components.
size_t group_bytes(long long cap);
Groups groups_of(char *buf, long long cap, int slot, int comp);
// Groups n blocks of block_bytes bytes (a multiple of 4; blocks 4-byte aligned) on stream s without synchronising:
// fingerprints keep their low hash_bits (0..64) bits, and every fingerprint match is confirmed byte for byte.  rep_out
// (may be nullptr) receives rep[i], the lowest index of a block byte-identical to block i.
int group_blocks(Handle *h, char *buf, long long cap, const uint8_t *blocks, int n, int block_bytes, int hash_bits,
                 int *rep_out, const Groups &g, cudaStream_t s);
// out[k] = blocks[distinct[k]], k < nd.
int gather_blocks(Handle *h, const uint8_t *blocks, const int *distinct, int nd, int block_bytes, uint8_t *out,
                  cudaStream_t s);
// For blocks i < n: hor | ver | dire (planes of `stride` blocks: 256, 256, 768 bytes each), flags and, when src_qt is
// given, the 64-byte qt map, from compact position slot[i] of the src arrays to position i of the dst arrays.
int expand_blocks(Handle *h, const int *slot, int n, long long stride, const uint8_t *src, uint8_t *dst,
                  const uint32_t *src_flags, uint32_t *dst_flags, const uint8_t *src_qt, uint8_t *dst_qt, cudaStream_t s);

}  // namespace pmp
