// Per-episode return-to-go scan fused with the window re-stack (SURVEY.md §2 K11).
//
// Restates label_reward.py:247-254 (discount_cumsum) and :232-245 (stack_outputs):
//   rtg[T-1] = r[T-1];  rtg[t] = r[t] + gamma * rtg[t+1]      strictly right-to-left, fp32, one add per step
//   out[i, f] = x[max(0, i - (F-1-f))]                         window left-padded with the episode's first value
// The scan's rounding is observable (SURVEY.md Appendix C), so the adds stay sequential inside an
// episode — parallelism is across episodes (one CTA each), across text groups (blockIdx.y: each group's
// rewards are scanned over the same episodes) and across the stacked writes.
// __fmul_rn/__fadd_rn forbid FMA contraction: numpy rounds the product before the add.
#pragma once

#include "common.cuh"

namespace arp {

constexpr int SCAN_THREADS = 128;
constexpr int SCAN_CHUNK = 2048;  // floats of one episode processed per smem pass

// reward [G,T] fp32; ep_off [n_eps+1] int64 (episode e = rows [ep_off[e], min(ep_off[e+1], T)));
// rtg [G,T] (optional), reward_stacked / rtg_stacked [G,T,F] (optional). Grid (n_eps, G): block (e, g) scans group g's
// slices of episode e.
__global__ void __launch_bounds__(SCAN_THREADS)
rtg_scan_stack_kernel(const float* __restrict__ reward, const long long* __restrict__ ep_off, long long T, int F,
                      float gamma, float* rtg, float* __restrict__ reward_stacked,
                      float* __restrict__ rtg_stacked) {
  __shared__ float s_r[SCAN_CHUNK + 64];
  __shared__ float s_g[SCAN_CHUNK + 64];
  __shared__ float s_carry;
  const int e = blockIdx.x;
  const long long lo = ep_off[e];
  const long long hi = min(ep_off[e + 1], T);
  if (hi <= lo) return;
  const int tid = threadIdx.x;
  {
    const long long gy = blockIdx.y;
    reward += gy * T;
    if (rtg) rtg += gy * T;
    if (reward_stacked) reward_stacked += gy * T * F;
    if (rtg_stacked) rtg_stacked += gy * T * F;
  }
  const float r_first = reward[lo];

  // walk the episode from its end in chunks; the running return crosses chunks through s_carry
  bool first_chunk = true;
  for (long long c_hi = hi; c_hi > lo; c_hi -= SCAN_CHUNK) {
    const long long c_lo = max(lo, c_hi - SCAN_CHUNK);
    const int n = static_cast<int>(c_hi - c_lo);
    // stage rewards [c_lo - (F-1), c_hi) so the stacked window of the chunk's first rows is in smem
    const int halo = static_cast<int>(min(static_cast<long long>(F - 1), c_lo - lo));
    for (int i = tid; i < n + halo; i += SCAN_THREADS) s_r[i + (F - 1 - halo)] = reward[c_lo - halo + i];
    __syncthreads();
    if (tid == 0) {
      float acc;
      int t = n - 1;
      if (first_chunk) {
        acc = s_r[F - 1 + t];
        s_g[F - 1 + t] = acc;
        --t;
      } else {
        acc = s_carry;
      }
      for (; t >= 0; --t) {
        acc = __fadd_rn(s_r[F - 1 + t], __fmul_rn(gamma, acc));
        s_g[F - 1 + t] = acc;
      }
      s_carry = acc;
    }
    __syncthreads();
    // rtg values for the halo rows are not known yet (they belong to the next, earlier chunk),
    // so rows whose window reaches into the halo are finished by that chunk: emit only complete rows.
    if (rtg)
      for (int i = tid; i < n; i += SCAN_THREADS) rtg[c_lo + i] = s_g[F - 1 + i];
    if (reward_stacked) {
      for (int i = tid; i < n * F; i += SCAN_THREADS) {
        const int row = i / F, f = i - row * F;
        const long long src = c_lo + row - (F - 1 - f);  // absolute index of the window element
        reward_stacked[(c_lo + row) * F + f] = src < lo ? r_first : s_r[F - 1 + row - (F - 1 - f)];
      }
    }
    first_chunk = false;
    __syncthreads();
  }
  // stacked rtg needs rtg of earlier rows, all of which are final only now: second sweep over global rtg.
  if (rtg_stacked) {
    const float* g = rtg;  // requires rtg != nullptr
    const long long n = hi - lo;
    const float g_first = g[lo];
    for (long long i = tid; i < n * F; i += SCAN_THREADS) {
      const long long row = i / F;
      const int f = static_cast<int>(i - row * F);
      const long long src = row - (F - 1 - f);
      rtg_stacked[(lo + row) * F + f] = src < 0 ? g_first : g[lo + src];
    }
  }
}

}  // namespace arp
