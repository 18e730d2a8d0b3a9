// latent.cuh -- generator latents z ~ N(0, 1) drawn on the device, bit-identical to
// `torch.randn((rows, Z), device='cuda', generator=g)` for a generator at Philox (seed, offset).
//
// torch's normal_ on CUDA (ATen/native/cuda/DistributionTemplates.h, distribution_elementwise_grid_stride_kernel with
// curand_normal4) fills a contiguous fp32 tensor of numel elements with
//     block = 256,  grid = min(num_SMs * (max_threads_per_SM / 256), ceil(numel / 256)),  T = 256 * grid
//     thread t: curand_init(seed, t, offset); round r = 0, 1, ...: one curand_normal4; component j of round r
//               goes to element e = r * 4T + j * T + t (when e < numel)
// and then advances the generator's offset by ((numel - 1) / 4T + 1) * 4.  Element e therefore depends only on
// (seed, offset, numel, e): any range of rows of a draw can be computed on its own.
//
// This kernel computes the same elements with one thread per (t, r) instead of a grid-stride loop over r: one
// Philox4x32-10 call, two Box-Muller pairs and four coalesced stores per thread.
//
// The Philox state, counter arithmetic and rounds are the toolkit's (curand_philox4x32_x.h).  curand_kernel.h itself
// is not included: it brings the XORWOW / MRG32k3a skip-ahead tables into the binary (+1.2 MB for this library).  So
// two short pieces of it are restated here, and must stay in step with it:
//   - curand_init(seed, t, offset) for offset % 4 == 0 (the only offsets torch's CUDA generator takes) is
//     ctr = (offset / 4, t), key = seed, and each curand4 / curand_normal4 call returns Philox(ctr) and then
//     increments ctr -- so round r uses Philox(ctr + r);
//   - curand_normal4 is _curand_box_muller (curand_normal.h) on (x, y) and (z, w).  Its expressions are copied
//     unchanged, so nvcc's default FMA contraction of x * 2^-32 + 2^-33 comes out as in torch's build.
#pragma once
#include <curand_globals.h>
#include <curand_philox4x32_x.h>
#include <stdint.h>

#include <algorithm>

namespace pbg {

constexpr int kLatentThreads = 256;   // torch's block size; also this kernel's

// The draw's grid-stride width T and the generator offset increment for a draw of numel elements.
struct LatentGeometry {
  long long T = 0;          // threads of torch's launch
  unsigned long long inc = 0;
};
inline LatentGeometry latent_geometry(long long numel, int num_sms, int max_threads_per_sm) {
  LatentGeometry g;
  const long long blocks = std::min<long long>(static_cast<long long>(num_sms) * (max_threads_per_sm / kLatentThreads),
                                               (numel + kLatentThreads - 1) / kLatentThreads);
  g.T = blocks * kLatentThreads;
  g.inc = static_cast<unsigned long long>((numel - 1) / (4 * g.T) + 1) * 4ull;
  return g;
}

// Device state of a ctx's latent stream: the Philox offset (the seed is a launch argument) and the finished-block
// counter of the launch that advances it.
struct LatentStream {
  unsigned long long offset;
  unsigned int done;
};

// _curand_box_muller, device branch (curand_normal.h)
__device__ __forceinline__ float2 latent_box_muller(unsigned int x, unsigned int y) {
  float2 result;
  float u = x * CURAND_2POW32_INV + (CURAND_2POW32_INV / 2);
  float v = y * CURAND_2POW32_INV_2PI + (CURAND_2POW32_INV_2PI / 2);
  float s = sqrtf(-2.0f * logf(u));
  __sincosf(v, &result.x, &result.y);
  result.x *= s;
  result.y *= s;
  return result;
}

struct LatentParams {
  unsigned long long seed;
  unsigned long long offset;      // used when st == nullptr; a multiple of 4
  LatentStream* st;               // the ctx's stream: offset read from here; advanced when `advance`
  int advance;                    // the last block to finish writes st->offset + inc
  unsigned long long inc;
  long long T;                    // torch's thread count for the whole draw
  long long e_begin, e_end;       // elements [e_begin, e_end) of the draw ...
  long long slot_begin;           // ... covered by threads (t, r) = slot % T, slot / T from slot_begin
  float* out;                     // [e_end - e_begin] fp32: element e at out[e - e_begin]
};

__global__ void __launch_bounds__(kLatentThreads) latent_draw_kernel(const LatentParams p) {
  const unsigned long long offset = p.st ? p.st->offset : p.offset;
  const long long slot = p.slot_begin + static_cast<long long>(blockIdx.x) * kLatentThreads + threadIdx.x;
  const long long t = slot % p.T, r = slot / p.T;
  const long long e0 = r * 4 * p.T + t;
  if (e0 < p.e_end && e0 + 3 * p.T >= p.e_begin) {
    curandStatePhilox4_32_10_t state;
    state.ctr = make_uint4(0, 0, 0, 0);
    state.key = make_uint2(static_cast<unsigned int>(p.seed), static_cast<unsigned int>(p.seed >> 32));
    Philox_State_Incr_hi(&state, static_cast<unsigned long long>(t));
    Philox_State_Incr(&state, offset / 4 + static_cast<unsigned long long>(r));
    const uint4 x = curand_Philox4x32_10(state.ctr, state.key);
    const float2 a = latent_box_muller(x.x, x.y), b = latent_box_muller(x.z, x.w);
    const float c[4] = {a.x, a.y, b.x, b.y};
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const long long e = e0 + j * p.T;
      // torch stores rand * std + mean with std = 1, mean = 0: the same value, except that -0 becomes +0
      if (e >= p.e_begin && e < p.e_end) p.out[e - p.e_begin] = __fadd_rn(c[j], 0.0f);
    }
  }
  if (p.st && p.advance) {
    __syncthreads();
    if (threadIdx.x == 0) {
      __threadfence();
      if (atomicAdd(&p.st->done, 1u) == gridDim.x - 1) {   // every other block has read the offset
        p.st->offset = offset + p.inc;
        p.st->done = 0;
        __threadfence();
      }
    }
  }
}

}  // namespace pbg
