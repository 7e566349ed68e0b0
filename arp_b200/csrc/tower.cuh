// The CLIP tower record of the adapter heads: what a fine-tuned adapter reads from the frozen CLIP tower, one fp32 row of
// TOWER_DIM = layers*W + E = 12*768 + 512 = 9728 columns per frame.
//   [0, layers*W)           the class-token taps, block l at [l*W, (l+1)*W): exactly the values the adapter's
//                           image_intermediate_linear GEMM multiplies (16-bit paths: ws.taps widened to fp32, which is
//                           exact; fp32 path: ws.taps32 as it is)
//   [layers*W, layers*W+E)  the un-normalised CLIP feature clip_head_kernel writes to featf[:, Dmid:]
// Fine-tuning freezes CLIP, so every adapter checkpoint of the same CLIP sees the same record: relabeling with a new
// adapter runs only the adapter tail (three GEMMs + the head) on it. tower_unpack_kernel narrows the taps back with
// pack_op, the conversion gather_cls_bf16_kernel uses, so the tail multiplies the very operand values of the frames path.
// Both kernels are memory-bound copies: one warp per frame row, 16-byte loads / stores.
#pragma once

#include "common.cuh"
#include "layernorm.cuh"   // load4_as_float

namespace arp {

constexpr int TOWER_TAPS = 12 * 768;
constexpr int TOWER_FEAT = 512;
constexpr int TOWER_DIM = TOWER_TAPS + TOWER_FEAT;   // 9728

__device__ __forceinline__ void store_tap4(float* p, float4 v) { *reinterpret_cast<float4*>(p) = v; }
__device__ __forceinline__ void store_tap4(op_t* p, float4 v) {
  *reinterpret_cast<uint2*>(p) = make_uint2(pack_op(v.x, v.y), pack_op(v.z, v.w));
}

// taps TT [>= n, TOWER_TAPS] (op_t: ws.taps, float: ws.taps32), feat fp32 [>= n, ld_feat] columns [feat_col0, +E)
//   -> rec fp32 [n, TOWER_DIM]
template <typename TT>
__global__ void __launch_bounds__(256)
tower_pack_kernel(const TT* __restrict__ taps, const float* __restrict__ feat, int ld_feat, int feat_col0,
                  float* __restrict__ rec, int n) {
  const int b = blockIdx.x * 8 + (threadIdx.x >> 5);
  if (b >= n) return;
  const int lane = threadIdx.x & 31;
  const TT* t = taps + static_cast<size_t>(b) * TOWER_TAPS;
  const float* f = feat + static_cast<size_t>(b) * ld_feat + feat_col0;
  float* r = rec + static_cast<size_t>(b) * TOWER_DIM;
#pragma unroll 4
  for (int c = lane * 4; c < TOWER_TAPS; c += 128) store_tap4(r + c, load4_as_float(t + c));
#pragma unroll
  for (int c = lane * 4; c < TOWER_FEAT; c += 128) store_tap4(r + TOWER_TAPS + c, load4_as_float(f + c));
}

// the inverse: rec fp32 [n, TOWER_DIM] -> taps TT [n, TOWER_TAPS], feat columns [feat_col0, +E) of rows [0, n)
template <typename TT>
__global__ void __launch_bounds__(256)
tower_unpack_kernel(const float* __restrict__ rec, TT* __restrict__ taps, float* __restrict__ feat, int ld_feat,
                    int feat_col0, int n) {
  const int b = blockIdx.x * 8 + (threadIdx.x >> 5);
  if (b >= n) return;
  const int lane = threadIdx.x & 31;
  const float* r = rec + static_cast<size_t>(b) * TOWER_DIM;
  TT* t = taps + static_cast<size_t>(b) * TOWER_TAPS;
  float* f = feat + static_cast<size_t>(b) * ld_feat + feat_col0;
#pragma unroll 4
  for (int c = lane * 4; c < TOWER_TAPS; c += 128) store_tap4(t + c, __ldg(reinterpret_cast<const float4*>(r + c)));
#pragma unroll
  for (int c = lane * 4; c < TOWER_FEAT; c += 128)
    store_tap4(f + c, __ldg(reinterpret_cast<const float4*>(r + TOWER_TAPS + c)));
}

}  // namespace arp
