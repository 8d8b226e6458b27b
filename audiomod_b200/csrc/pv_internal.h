// Internals shared by the translation units of libpvgpu.so (not part of the C ABI).
#pragma once
#include <cstddef>
#include <cstdint>
#include <string>

namespace pvgpu {
// Sets the calling thread's pvgpu_last_error() message and returns `code`.
int fail(int code, const char *fmt, ...);
// Message of the calling thread (worker threads hand theirs to the thread that called the C ABI).
const std::string &last_error_string();
// memcpy of floats with non-temporal stores (pv_multi.cc): for page-locked staging blocks a DMA engine reads next -- lines
// left dirty in several cores' caches made the host-to-device copy run at 7..14 GB/s instead of 50 (scripts/h2d_dirty_probe.py).
// Call copy_nt_fence() once after a batch of copies, on the thread that made them.
void copy_nt(float *dst, const float *src, size_t n);
// the same for int16 samples (live batches of int16 rows); a destination on a 2-byte boundary takes one plain store first
void copy_nt(int16_t *dst, const int16_t *src, size_t n);
void copy_nt_fence();
}  // namespace pvgpu
