// Host-side helpers of libavrf_gpu.so (hostutil.cpp).
#pragma once
#include <stddef.h>
#include <stdint.h>

namespace avrf {
// Copy into the pinned staging buffers of single pushes with non-temporal stores (32-byte multiples into 32-byte
// aligned destinations; plain memcpy otherwise): the staged bytes are read next by the GPU's DMA engine, not by
// this core, so they need not displace the caller's working set or cost a read-for-ownership.
void stage_copy(void* dst, const void* src, size_t n);
// One fixed-size field of a staged proof: `bytes` (a multiple of 32) from `src` to the 32-byte aligned `dst`.
struct StageField {
  uint8_t* dst;
  const uint8_t* src;
  size_t bytes;
};
// One proof of a single push into the staging arrays, one call: its `nf` fields, then `io_bytes` of I/O pairs into the
// 32-byte aligned `dio`.
void stage_proof(const StageField* f, size_t nf, uint8_t* dio, const uint8_t* ios, size_t io_bytes);
// Orders the non-temporal stores before the DMA is queued.
void stage_fence();
}  // namespace avrf
