// Counter-based dropout masks (maxvit.py:146,151: nn.Dropout on the attention probabilities and after to_out).
// A mask byte is a pure function of (seed, row id, group id), so the forward kernel, the backward kernels and the test
// oracle regenerate identical masks without storing them.  One 32-bit hash yields four mask bytes; an element is kept
// when its byte >= T, i.e. the drop probability is quantised to p_eff = T / 256 and kept values are scaled by 256 / (256 - T).
#pragma once
#include <stdint.h>

namespace vg {

__host__ __device__ __forceinline__ uint32_t drop_hash(uint32_t seed, uint32_t a, uint32_t b) {
  uint32_t x = a * 0x9E3779B1u + b * 0x85EBCA77u + seed;
  x ^= x >> 16; x *= 0x85EBCA6Bu; x ^= x >> 13; x *= 0xC2B2AE35u; x ^= x >> 16;
  return x;
}
// group ids: attention probabilities of (head h, keys 4g..4g+3), g in [0,16) (windows of up to 64 tokens, see drop_slots);
// to_out outputs of channels 4g..4g+3
__host__ __device__ __forceinline__ uint32_t drop_group_prob(uint32_t salt, int h, int g) { return salt * 8192u + (uint32_t)h * 16u + (uint32_t)g; }
__host__ __device__ __forceinline__ uint32_t drop_group_out(uint32_t salt, int g) { return salt * 8192u + 4096u + (uint32_t)g; }
// row id of token slot i (0..63) of window wdx
__host__ __device__ __forceinline__ uint32_t drop_row(long long wdx, int i) { return (uint32_t)(wdx * 64 + i); }

// Windows of 65 .. 128 tokens (the un-fused path only) double both strides, so that no two (window, token) rows or (head, key
// group) pairs share a counter: 128 slots per window, 32 key groups per head.  The probability ids salt*8192 + h*32 + g stay
// below the to_out range salt*8192 + 4096 only for heads <= 128, which the entry points check.  Windows of up to 64 tokens keep
// the ids above (slots = 64), so their masks are the same as the fused kernels'.
__host__ __device__ __forceinline__ int drop_slots(int S) { return S > 64 ? 128 : 64; }
__host__ __device__ __forceinline__ uint32_t drop_row(long long wdx, int i, int slots) { return (uint32_t)(wdx * slots + i); }
__host__ __device__ __forceinline__ uint32_t drop_group_prob(uint32_t salt, int h, int g, int slots) {
  return salt * 8192u + (uint32_t)h * (uint32_t)(slots / 4) + (uint32_t)g;
}
constexpr int DROP_MAX_HEADS_LONG = 128;   // heads limit of 128-slot probability dropout

struct DropCfg {
  uint32_t seed, salt;
  int thresh;          // 0 = no dropout
  float scale;         // 256 / (256 - thresh)
};

}  // namespace vg
