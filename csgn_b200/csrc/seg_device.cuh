// seg_device.cuh -- device helpers of the ciphertext-array kernels (segments.cu) and the circuit kernel (circuit.cu):
// unit-wise AND, popcount and equality over 8-byte (uint2) and 16-byte (uint4) units, and the block hash of the
// cancellation.  Internal: each translation unit gets its own copy (anonymous namespace).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

namespace csgn {
namespace {

__device__ __forceinline__ uint4 vand(const uint4 x, const uint4 y) {
    return make_uint4(x.x & y.x, x.y & y.y, x.z & y.z, x.w & y.w);
}
__device__ __forceinline__ uint2 vand(const uint2 x, const uint2 y) { return make_uint2(x.x & y.x, x.y & y.y); }
__device__ __forceinline__ uint32_t vpopc(const uint4 x) { return __popc(x.x) + __popc(x.y) + __popc(x.z) + __popc(x.w); }
__device__ __forceinline__ uint32_t vpopc(const uint2 x) { return __popc(x.x) + __popc(x.y); }

// A block's hash is the splitmix64 finaliser of the sum of its words' finalised values (each word offset by its
// position), so the lanes that hold a block's units add their parts in any order.
__device__ __forceinline__ uint64_t mix64(uint64_t x) {
    x ^= x >> 30;
    x *= 0xbf58476d1ce4e5b9ull;
    x ^= x >> 27;
    x *= 0x94d049bb133111ebull;
    return x ^ (x >> 31);
}
__device__ __forceinline__ uint64_t word_hash(uint64_t x, uint64_t w) { return mix64(x + (w + 1) * 0x9e3779b97f4a7c15ull); }
__device__ __forceinline__ uint64_t unit_hash(const uint2 u, uint32_t w) {
    return word_hash((uint64_t)u.y << 32 | u.x, w);
}
__device__ __forceinline__ uint64_t unit_hash(const uint4 u, uint32_t w) {
    return word_hash((uint64_t)u.y << 32 | u.x, 2ull * w) + word_hash((uint64_t)u.w << 32 | u.z, 2ull * w + 1);
}
__device__ __forceinline__ bool veq(const uint2 x, const uint2 y) { return x.x == y.x && x.y == y.y; }
__device__ __forceinline__ bool veq(const uint4 x, const uint4 y) {
    return x.x == y.x && x.y == y.y && x.z == y.z && x.w == y.w;
}

}  // namespace
}  // namespace csgn
