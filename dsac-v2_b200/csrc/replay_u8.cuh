// Replay gather for 8-bit image rings (dsact_cnn_replay_bind_u8, include/dsact.h).  The ring stores every pixel of
// obs / obs2 as its code k in [0, 255]; the pixel is float32(k) / 255.0f, correctly rounded.  That is the value the
// reference's pixel environments produce (rgb / 255 in float64, then cast), for all 256 codes.  A reciprocal multiply
// (k * (1/255)) is wrong for about half of them, so the 256 pixel values come from __fdiv_rn, which stays IEEE
// round-to-nearest under --use_fast_math.  Every block fills a shared-memory table with them once and decodes by lookup
// (a division per pixel made the gather slower than the fp32 one).  The gathered minibatch is the fp32 arena
// gather_kernel writes, with the same values.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "kernels.cuh"

namespace dsact {

constexpr int GATHER_U8_THREADS = 64;   // two rows per block: small batches still spread over most SMs

// the four codes of one 32-bit word, lowest byte first (the byte order of the row), through the block's table
__device__ __forceinline__ float4 decode_u8x4(const float* lut, uint32_t w) {
  return make_float4(lut[w & 0xffu], lut[(w >> 8) & 0xffu], lut[(w >> 16) & 0xffu], lut[w >> 24]);
}

// decode the image rows of obs and obs2 (O codes each, at s[0] / s[1]) into O floats each at d[0] / d[1]; the lanes of a
// warp split the rows
__device__ __forceinline__ void decode_rows_u8(const float* lut, const uint8_t* const (&s)[2], float* const (&d)[2], int O, int lane) {
  if ((O & 15) == 0) {
    // 16 codes per lane and load, two loads of obs and two of obs2 in flight per lane (the gather is bound by DRAM
    // latency on random rows); four float4 stores per load
    const int n16 = O >> 4;
    for (int c0 = lane; c0 < n16; c0 += 64) {
      uint4 w[2][2];
#pragma unroll
      for (int u = 0; u < 2; ++u)
#pragma unroll
        for (int t = 0; t < 2; ++t)
          if (c0 + 32 * u < n16) w[t][u] = __ldg(reinterpret_cast<const uint4*>(s[t]) + c0 + 32 * u);
#pragma unroll
      for (int u = 0; u < 2; ++u) {
        const int c = c0 + 32 * u;
        if (c < n16) {
#pragma unroll
          for (int t = 0; t < 2; ++t) {
            float4* d4 = reinterpret_cast<float4*>(d[t]) + 4 * c;
            d4[0] = decode_u8x4(lut, w[t][u].x);
            d4[1] = decode_u8x4(lut, w[t][u].y);
            d4[2] = decode_u8x4(lut, w[t][u].z);
            d4[3] = decode_u8x4(lut, w[t][u].w);
          }
        }
      }
    }
  } else if ((O & 3) == 0) {   // rows start on 4-byte boundaries (ring) and on 16-byte boundaries (arena)
    for (int c = lane; c < (O >> 2); c += 32) {
      const uint32_t a = __ldg(reinterpret_cast<const uint32_t*>(s[0]) + c), b = __ldg(reinterpret_cast<const uint32_t*>(s[1]) + c);
      reinterpret_cast<float4*>(d[0])[c] = decode_u8x4(lut, a);
      reinterpret_cast<float4*>(d[1])[c] = decode_u8x4(lut, b);
    }
  } else {   // odd row lengths (e.g. 3x13x11 = 429 bytes): rows start at any byte
    for (int c = lane; c < O; c += 32) {
      d[0][c] = lut[__ldg(s[0] + c)];
      d[1][c] = lut[__ldg(s[1] + c)];
    }
  }
}

// gather_kernel's contract (training/replay_buffer.py:87-90) on a ring with uint8 obs / obs2: one warp per sampled row.
// draw_idx != null: no index list was given; every warp draws its row's index with gather_kernel's Philox stream
// (replay_index: same seed, same counter, same rows), so an fp32 ring and an 8-bit ring holding the same transitions
// sample the same minibatch.  rng_advance_kernel steps the counter afterwards, as for gather_kernel.
__global__ void gather_u8_kernel(const uint8_t* __restrict__ r_obs, const uint8_t* __restrict__ r_obs2,
                                 const float* __restrict__ r_act, const float* __restrict__ r_rew,
                                 const float* __restrict__ r_done, const float* __restrict__ r_logp,
                                 const int64_t* __restrict__ idx, float* __restrict__ obs, float* __restrict__ obs2,
                                 float* __restrict__ act, float* __restrict__ rew, float* __restrict__ done,
                                 float* __restrict__ logp, int B, int O, int A, int64_t* __restrict__ draw_idx, uint64_t seed,
                                 const float* __restrict__ state) {
  pdl_sync();
  __shared__ float lut[256];
  for (int k = threadIdx.x; k < 256; k += blockDim.x) lut[k] = __fdiv_rn(__uint2float_rn((uint32_t)k), 255.0f);
  __syncthreads();
  const int lane = threadIdx.x & 31;
  const int wpb = blockDim.x >> 5;
  uint32_t step = 0;
  int64_t size = 1;
  const uint2 key = make_uint2((uint32_t)seed, (uint32_t)(seed >> 32));
  if (draw_idx) {
    step = reinterpret_cast<const uint32_t*>(state)[ST_RNG_CTR];
    size = *reinterpret_cast<const int64_t*>(state + ST_RB_SIZE);
  }
  for (int row = blockIdx.x * wpb + (threadIdx.x >> 5); row < B; row += gridDim.x * wpb) {
    int64_t src;
    if (draw_idx) {
      src = replay_index(row, step, size, key);
      if (lane == 0) draw_idx[row] = src;
    } else {
      src = idx[row];
    }
    const uint8_t* const s[2] = {r_obs + src * O, r_obs2 + src * O};
    float* const d[2] = {obs + (size_t)row * O, obs2 + (size_t)row * O};
    decode_rows_u8(lut, s, d, O, lane);
    for (int c = lane; c < A; c += 32) act[(size_t)row * A + c] = __ldg(r_act + src * A + c);
    if (lane == 0) { rew[row] = __ldg(r_rew + src); done[row] = __ldg(r_done + src); logp[row] = __ldg(r_logp + src); }
  }
}

}  // namespace dsact
