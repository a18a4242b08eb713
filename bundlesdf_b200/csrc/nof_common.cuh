// Shared device/host helpers for libnof_sm100 (sm_100a only).
#pragma once
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/nof.h"

namespace nof {

void set_error(const char* fmt, ...);
int check_launch(const char* what);

#define NOF_REQUIRE(cond, ...)            \
  do {                                    \
    if (!(cond)) {                        \
      nof::set_error(__VA_ARGS__);        \
      return NOF_E_INVALID;               \
    }                                     \
  } while (0)

static inline cudaStream_t as_stream(nof_stream_t s) { return reinterpret_cast<cudaStream_t>(s); }

template <typename T>
static inline __host__ __device__ T div_up(T a, T b) { return (a + b - 1) / b; }

// ---------------------------------------------------------------------------------------------------
// Hash-grid level geometry. Bit-for-bit the reference's device arithmetic (gridencoder.cu:155-156):
//   scale = exp2f(level * S) * H - 1.0f   (nvcc contracts the mul+sub into one FMA)
//   resolution = (uint32_t)ceil(scale) + 1
// ---------------------------------------------------------------------------------------------------
struct LevelGeom {
  float scale;
  uint32_t resolution;
  uint32_t hashmap_size;
  uint32_t offset;      // entries
  uint32_t dense;       // 1 if the dense (strided) index is used for D=3, else hashed
};

__device__ __forceinline__ float level_scale(uint32_t level, float S, uint32_t H) {
  return __fmaf_rn(exp2f((float)level * S), (float)H, -1.0f);
}

__device__ __forceinline__ LevelGeom level_geom3(uint32_t level, float S, uint32_t H, const int32_t* __restrict__ offsets) {
  LevelGeom g;
  g.scale = level_scale(level, S, H);
  g.resolution = (uint32_t)ceilf(g.scale) + 1u;
  g.offset = (uint32_t)offsets[level];
  g.hashmap_size = (uint32_t)offsets[level + 1] - g.offset;
  // gridencoder.cu:66-83 for D=3, align_corners=false: the loop multiplies stride by (res+1) while
  // stride <= hashmap_size; hashing happens iff the final stride exceeds hashmap_size.
  uint64_t r1 = (uint64_t)g.resolution + 1u;
  uint32_t stride = 1;
  for (int d = 0; d < 3 && stride <= g.hashmap_size; ++d) stride *= (uint32_t)r1;   // uint32 wrap like the reference
  g.dense = !(stride > g.hashmap_size);
  return g;
}

// gridencoder.cu:47-83 — index of one grid corner (D=3, align_corners=false).
__device__ __forceinline__ uint32_t grid_index3(uint32_t gridtype, uint32_t hashmap_size, uint32_t resolution,
                                                uint32_t x, uint32_t y, uint32_t z) {
  uint32_t stride = 1, index = 0;
  const uint32_t r1 = resolution + 1u;
  if (stride <= hashmap_size) { index += x * stride; stride *= r1; }
  if (stride <= hashmap_size) { index += y * stride; stride *= r1; }
  if (stride <= hashmap_size) { index += z * stride; stride *= r1; }
  if (gridtype == 0 && stride > hashmap_size) index = (x * 1u) ^ (y * 2654435761u) ^ (z * 805459861u);
  return index % hashmap_size;
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// vectorised fp32 reduction (no return value): red.global.add.v2.f32 is sm_90+.
__device__ __forceinline__ void red_add_v2(float* addr, float a, float b) {
  asm volatile("red.global.add.v2.f32 [%0], {%1, %2};" ::"l"(addr), "f"(a), "f"(b) : "memory");
}
// 16-byte form: same L2 atomic-unit cost per lane as the 4- and 8-byte forms (profiles/red_bench.cu: ~180 G lane-ops/s for
// random addresses whatever the width), so two adjacent table entries in one op halve the cost.
__device__ __forceinline__ void red_add_v4(float* addr, float a, float b, float c, float d) {
  asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(addr), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}
__device__ __forceinline__ void red_add(float* addr, float a) {
  asm volatile("red.global.add.f32 [%0], %1;" ::"l"(addr), "f"(a) : "memory");
}

// Philox4x32-10 counter RNG -> uniform [0,1) floats (same construction torch / curand use; the stream itself is
// ours: tests/test_gpu_ray_march.py pins the ray march's draws to a numpy restatement checked on the Random123 vectors).
__device__ __forceinline__ uint4 philox4x32_10(uint4 ctr, uint2 key) {
  const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
  for (int i = 0; i < 10; ++i) {
    uint32_t hi0 = __umulhi(M0, ctr.x), lo0 = M0 * ctr.x;
    uint32_t hi1 = __umulhi(M1, ctr.z), lo1 = M1 * ctr.z;
    ctr = make_uint4(hi1 ^ ctr.y ^ key.x, lo1, hi0 ^ ctr.w ^ key.y, lo0);
    key.x += W0;
    key.y += W1;
  }
  return ctr;
}
__device__ __forceinline__ float u32_to_unit(uint32_t x) { return (float)(x >> 8) * (1.0f / 16777216.0f); }

}  // namespace nof
