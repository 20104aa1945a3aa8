// Keras Dropout(rate) between BatchNormalization and the activation of a dense block: the one mask function of the
// library.  Every kernel that applies the dropout calls dropout_keep4; tests/dropout_ref.py restates it in NumPy.
//
// The keep bit of element (row, col) of dense block `block` in training step `step` under seed `seed`:
//   u    = word (col & 3) of Philox4x32-10(ctr = (col >> 2, row, block, step lo32), key = (seed lo32, seed hi32))
//   keep = u >= threshold,  threshold = (uint32) min(floor(rate * 2^32), 2^32 - 1)
// and a kept element is multiplied by scale = (float)(1 / (1 - rate)).  The mask is a function of (seed, step, block,
// row, column) only - not of the kernel, thread mapping or batch bucket that evaluates it - so the forward, the backward
// and the reference agree bit for bit without storing it.  threshold and scale are formed on the host in double
// (model.cu: make_dropout).
#pragma once
#include <stdint.h>

#include <curand_philox4x32_x.h>

namespace gcs {

struct Dropout {
  uint32_t threshold;   // 0: no dropout (every element kept with scale 1)
  float scale;
  uint64_t seed;
  uint32_t step;        // low 32 bits of the step counter
  int32_t block;        // index of the dense block (params.py block order)
};

// Keep bits of columns 4q .. 4q+3 of `row` (bit k = column 4q + k).
__device__ __forceinline__ unsigned dropout_keep4(const Dropout& d, int64_t row, int q) {
  const uint4 ctr = make_uint4(static_cast<uint32_t>(q), static_cast<uint32_t>(row), static_cast<uint32_t>(d.block), d.step);
  const uint2 key = make_uint2(static_cast<uint32_t>(d.seed), static_cast<uint32_t>(d.seed >> 32));
  const uint4 u = curand_Philox4x32_10(ctr, key);
  return (u.x >= d.threshold ? 1u : 0u) | (u.y >= d.threshold ? 2u : 0u) | (u.z >= d.threshold ? 4u : 0u) |
         (u.w >= d.threshold ? 8u : 0u);
}

// m * scale * y with m the keep bit `k` of `bits`.
__device__ __forceinline__ float dropout_apply(const Dropout& d, unsigned bits, int k, float y) {
  return (bits >> k) & 1u ? y * d.scale : 0.f;
}

}  // namespace gcs
