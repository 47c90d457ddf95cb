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

}  // namespace pmp
