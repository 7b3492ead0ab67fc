// block_select.cuh — an exact order statistic over the float bits of one block's values (cv ICP mode's median / MAD,
// the median and trimmed correspondence rejectors of the PCL ICP).
#pragma once

#include <cuda_runtime.h>

namespace peb {

// exact order statistic `nth` of m non-negative floats f(i), by three radix passes over the float bits (11 + 11 + 10);
// one block of 1024 threads; returns the value to every thread.  The result is the nth of the taken values ordered by
// their bit patterns (for non-negative floats, +inf and denormals included, their numeric order).
// Precondition: nth < (number of values taken).  Outside it no bin holds the rank and the bin state read after the
// scan is whatever an earlier pass or call left in shared memory.
// SKIP_NEG: values with the sign bit set are not taken (how a caller leaves entries out); the values of the others
// and nth then refer to the taken ones only.  -0.0f has the sign bit and is skipped as well.
template <typename F, bool SKIP_NEG = false>
__device__ float block_select_nth(F f, int m, int nth, unsigned* hist /* shared [2048] */, unsigned* s_state /* shared [2] */,
                                  unsigned* s_wsum /* shared [32] */) {
  unsigned prefix = 0u, prefix_mask = 0u;
  int want = nth;
  const int shifts[3] = {21, 10, 0};
  const int bits[3] = {11, 11, 10};
  for (int pass = 0; pass < 3; ++pass) {
    const int nb = 1 << bits[pass];
    for (int b = threadIdx.x; b < nb; b += blockDim.x) hist[b] = 0u;
    __syncthreads();
    for (int i = threadIdx.x; i < m; i += blockDim.x) {
      const unsigned u = __float_as_uint(f(i));
      const bool in = (u & prefix_mask) == prefix && (!SKIP_NEG || (u >> 31) == 0u);
      // distances cluster in a few bins: lanes that hit the same bin add once (the loop bound is warp-uniform up to the tail)
      const unsigned act = __ballot_sync(__activemask(), in);
      if (in) {
        const unsigned bin = (u >> shifts[pass]) & (nb - 1);
        const unsigned peers = __match_any_sync(act, bin);
        if ((threadIdx.x & 31) == static_cast<unsigned>(__ffs(peers) - 1)) atomicAdd(&hist[bin], static_cast<unsigned>(__popc(peers)));
      }
    }
    __syncthreads();
    {
      // the bin that holds the wanted rank: block-wide prefix sum over the bins (blockDim.x = 1024 threads, 1 or 2 bins each)
      const int per = nb / static_cast<int>(blockDim.x);
      unsigned local = 0u;
      for (int k = 0; k < per; ++k) local += hist[threadIdx.x * per + k];
      const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
      unsigned x = local;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const unsigned y = __shfl_up_sync(0xFFFFFFFFu, x, o);
        if (lane >= o) x += y;
      }
      if (lane == 31) s_wsum[warp] = x;
      __syncthreads();
      if (warp == 0) {
        unsigned w = s_wsum[lane];
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
          const unsigned y = __shfl_up_sync(0xFFFFFFFFu, w, o);
          if (lane >= o) w += y;
        }
        s_wsum[lane] = w;
      }
      __syncthreads();
      const unsigned before = x - local + (warp ? s_wsum[warp - 1] : 0u);
      const unsigned w = static_cast<unsigned>(want);
      if (w >= before && w < before + local) {
        unsigned acc = before;
        for (int k = 0; k < per; ++k) {
          const unsigned c = hist[threadIdx.x * per + k];
          if (acc + c > w) {
            s_state[0] = static_cast<unsigned>(threadIdx.x * per + k);
            s_state[1] = w - acc;
            break;
          }
          acc += c;
        }
      }
    }
    __syncthreads();
    prefix |= s_state[0] << shifts[pass];
    prefix_mask |= static_cast<unsigned>(nb - 1) << shifts[pass];
    want = static_cast<int>(s_state[1]);
    __syncthreads();
  }
  return __uint_as_float(prefix);
}

}  // namespace peb
