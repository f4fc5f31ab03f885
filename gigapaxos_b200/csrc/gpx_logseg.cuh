/*
 * gpx_logseg.cuh -- the size of a log segment (format: include/gpx.h:187-209), stated once for the kernels that
 * write segments and for the host that checks a call against the ring and mirrors the ring heads.
 *
 * A segment is a 64-byte header, one record image per slot (48 B for an ACCEPT, 32 B for a DECISION or a PREPARE)
 * and, in an ACCEPT segment, a payload area; the segment is padded to a multiple of 32 bytes.
 */
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

__host__ __device__ __forceinline__ unsigned long long seg_align32(unsigned long long x) { return (x + 31ull) & ~31ull; }
/* offset of an ACCEPT segment's payload area from the segment start */
__host__ __device__ __forceinline__ unsigned long long seg_pay_rel(uint32_t n) {
  return 64ull + (unsigned long long)n * 48ull;
}
/* an ACCEPT segment of n images and pay_bytes of payload area */
__host__ __device__ __forceinline__ unsigned long long seg_accept_bytes(uint32_t n, unsigned long long pay_bytes) {
  return seg_align32(seg_pay_rel(n) + pay_bytes);
}
/* a DECISION or PREPARE segment of n images */
__host__ __device__ __forceinline__ unsigned long long seg_decision_bytes(uint32_t n) {
  return 64ull + (unsigned long long)n * 32ull;
}
