// Reward heads (SURVEY.md §2 K9 / K10 epilogues): everything after the last resblock, fused per frame.
//
//  clip head      f = ln_post(x[:,0]) @ proj ; reward = exp(logit_scale) * <f/|f|, t/|t|>
//                 (openai/CLIP VisionTransformer tail + CLIP.forward, called at label_reward.py:141-145)
//  adapter head   a = sigma(w) * feat + (1 - sigma(w)) * mlp(feat) ; L2-normalise ; same cosine
//                 (finetune_module/clip_multiscale_adapter.py:145-151, label_reward.py:213-228);
//                 "ensemble" variant normalises each of the 13 512-wide scales separately and
//                 averages the 13 cosines (label_reward.py:217-222).
//  Text embeddings arrive already L2-normalised (cached once per run; the reference re-runs the
//  text tower every episode, label_reward.py:135-138). All n_text cosines are produced; `reduce`
//  picks row 0 (what the reference actually does — SURVEY.md Q1) or the mean.
//  Text groups: the n_text rows are the concatenation of G instruction sets, group g = rows
//  [group_off[g], group_off[g+1]), and each group is reduced on its own into reward[g * ld + frame]. A group's
//  reward is bit-identical to a call with that group's rows alone: every cosine is a warp dot product whose order does
//  not depend on the text's index, and `reduce` accumulates in text order from the group's first row, then divides by
//  the group size.
//  Stored embeddings: the per-frame vector the instruction side starts from (clip: f before normalisation; adapter: the
//  gated a) can be kept and relabeled later without frames or image weights — clip_embedding_head_kernel, and
//  adapter_head_kernel with mlp == nullptr. They run the same instruction-side code as the frames path, so the rewards
//  are bit-identical.
// fp32 throughout: these are a few hundred KFLOP per frame, L2-resident weights.
#pragma once

#include "common.cuh"

namespace arp {

constexpr int HEAD_MAX_TEXT = 16;         // texts of one group
constexpr int HEAD_MAX_GROUPS = 16;       // groups of one call
constexpr int HEAD_MAX_TEXT_TOTAL = 64;   // texts of all groups together
enum HeadReduce : int { REDUCE_FIRST = 0, REDUCE_MEAN = 1 };

template <int NT>
__device__ __forceinline__ float block_sum(float v, float* scratch) {
  // all NT threads call; returns the total to every thread
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  v = warp_sum(v);
  __syncthreads();
  if (lane == 0) scratch[warp] = v;
  __syncthreads();
  float t = 0.f;
#pragma unroll
  for (int i = 0; i < NT / 32; ++i) t += scratch[i];
  return t;
}

constexpr int HEAD_FR = 4;
constexpr int HEAD_SMEM_BYTES = 8 * HEAD_FR * 512 * 4;   // dynamic: the per-warp partial outputs of clip_head_kernel

// The instruction side of the clip head, shared by clip_head_kernel (features projected from the class-token rows) and
// clip_embedding_head_kernel (stored features): s_y[f] holds frame b0+f's un-normalised feature (zeros past nf); thread
// tid owns columns tid + j*256 of every row. Both kernels run this same code, so the same FMA contractions happen and a
// stored embedding relabels to the bits of the frames path.
template <int E>
__device__ __forceinline__ void clip_head_cosines(float (*s_y)[E], float* s_red, float* s_inv,
                                                  float (*s_logit)[HEAD_MAX_TEXT_TOTAL], int b0, int nf,
                                                  const float* __restrict__ text, int n_text,
                                                  const int* __restrict__ group_off, int n_groups, float scale,
                                                  int reduce, float* __restrict__ logits, float* __restrict__ reward,
                                                  long long ld) {
  const int tid = threadIdx.x;
  if (text == nullptr) return;
  for (int f = 0; f < HEAD_FR; ++f) {
    float n2 = 0.f;
#pragma unroll
    for (int j = 0; j < E / 256; ++j) {
      const float yv = s_y[f][tid + j * 256];
      n2 += yv * yv;
    }
    const float tot = block_sum<256>(n2, s_red);
    if (tid == 0) s_inv[f] = 1.0f / sqrtf(tot);
  }
  __syncthreads();

  // cosines: warp w handles (frame, text) pairs w, w+8, ...
  const int warp = tid >> 5, lane = tid & 31;
  for (int p = warp; p < nf * n_text; p += 8) {
    const int f = p / n_text, t = p - f * n_text;
    float d = 0.f;
    for (int k = lane; k < E; k += 32) d = fmaf(s_y[f][k], __ldg(text + static_cast<size_t>(t) * E + k), d);
    d = warp_sum(d);
    if (lane == 0) {
      const float lg = scale * (d * s_inv[f]);
      s_logit[f][t] = lg;
      if (logits) logits[static_cast<size_t>(b0 + f) * n_text + t] = lg;
    }
  }
  __syncthreads();
  if (tid < nf * n_groups && reward) {       // thread -> (group, frame)
    const int g = tid / nf, f = tid - g * nf;
    const int t0 = group_off[g], t1 = group_off[g + 1];
    float r = s_logit[f][t0];
    if (reduce == REDUCE_MEAN) {
      for (int t = t0 + 1; t < t1; ++t) r += s_logit[f][t];
      r /= static_cast<float>(t1 - t0);
    }
    reward[g * ld + b0 + f] = r;
  }
}

// One CTA (256 threads) per FR consecutive frames: the 768x512 projection is streamed once per CTA and applied to all
// FR class-token rows (with one frame per CTA the 1.5 MB matrix was re-read from L2 by every CTA).
//   x        fp32 [B*tokens, W]   residual stream after the last block (row b*tokens = class token)
//   proj     fp32 [W, E]
//   text     fp32 [n_text, E] unit rows of all groups (may be null when only features are wanted)
//   group_off int32 [n_groups + 1] row offsets of the groups into text
//   feat_out fp32 [B, ld_feat] : un-normalised f written at column feat_col0 (adapter / goal modes) or null
//   logits   fp32 [B, n_text] or null ; reward fp32 [n_groups, ld] (group-major, frame b at column b) or null
template <int W, int E>
__global__ void __launch_bounds__(256)
clip_head_kernel(const float* __restrict__ x, int tokens, const float* __restrict__ ln_g,
                 const float* __restrict__ ln_b, float eps, const float* __restrict__ proj,
                 const float* __restrict__ text, int n_text, const int* __restrict__ group_off, int n_groups,
                 float scale, int reduce, float* __restrict__ feat_out, int ld_feat, int feat_col0,
                 float* __restrict__ logits, float* __restrict__ reward, long long ld, int n_frames) {
  static_assert(W % 256 == 0 && E % 256 == 0, "head widths must be multiples of the CTA size");
  __shared__ float s_f[HEAD_FR][W];
  __shared__ float s_y[HEAD_FR][E];
  __shared__ float s_red[8];
  __shared__ float s_inv[HEAD_FR];
  __shared__ float s_logit[HEAD_FR][HEAD_MAX_TEXT_TOTAL];
  const int b0 = blockIdx.x * HEAD_FR, tid = threadIdx.x;
  const int nf = min(HEAD_FR, n_frames - b0);

  for (int f = 0; f < HEAD_FR; ++f) {        // ln_post of each class-token row (zeros for frames past the end)
    float v[W / 256];
    float s = 0.f;
    if (f < nf) {
      const float* xr = x + static_cast<size_t>(b0 + f) * tokens * W;
#pragma unroll
      for (int i = 0; i < W / 256; ++i) { v[i] = xr[tid + i * 256]; s += v[i]; }
    } else {
#pragma unroll
      for (int i = 0; i < W / 256; ++i) v[i] = 0.f;
    }
    const float mean = block_sum<256>(s, s_red) * (1.0f / W);
    float q = 0.f;
#pragma unroll
    for (int i = 0; i < W / 256; ++i) { const float d = v[i] - mean; q += d * d; }
    const float rstd = rsqrtf(block_sum<256>(q, s_red) * (1.0f / W) + eps);
#pragma unroll
    for (int i = 0; i < W / 256; ++i) {
      const int c = tid + i * 256;
      s_f[f][c] = f < nf ? (v[i] - mean) * rstd * ln_g[c] + ln_b[c] : 0.f;
    }
  }
  __syncthreads();

  // projection, split over k across the 8 warps: a warp streams whole 2 KB rows of proj (4 x LDG.128 per lane, 16 loads
  // in flight) for its 96 values of k and keeps FR x 16 partial outputs per lane; the partials meet in shared memory.
  // (One output pair per thread over all 768 k was a chain of 192 dependent L2 round trips: ~100 us per CTA.)
  static_assert(E == 512 && W % 8 == 0, "lane -> column mapping below assumes 512 outputs");
  extern __shared__ float s_part[];            // [8 warps][HEAD_FR][E]
  {
    const int warp = tid >> 5, lane = tid & 31;
    constexpr int KW = W / 8;
    float acc[HEAD_FR][16];
#pragma unroll
    for (int f = 0; f < HEAD_FR; ++f)
#pragma unroll
      for (int j = 0; j < 16; ++j) acc[f][j] = 0.f;
    const float4* prow = reinterpret_cast<const float4*>(proj) + static_cast<size_t>(warp) * KW * (E / 4) + lane;
#pragma unroll 4
    for (int kk = 0; kk < KW; ++kk) {
      float4 pv[4];
#pragma unroll
      for (int g = 0; g < 4; ++g) pv[g] = __ldg(prow + static_cast<size_t>(kk) * (E / 4) + g * 32);
#pragma unroll
      for (int f = 0; f < HEAD_FR; ++f) {
        const float fk = s_f[f][warp * KW + kk];
#pragma unroll
        for (int g = 0; g < 4; ++g) {
          acc[f][4 * g] = fmaf(fk, pv[g].x, acc[f][4 * g]);
          acc[f][4 * g + 1] = fmaf(fk, pv[g].y, acc[f][4 * g + 1]);
          acc[f][4 * g + 2] = fmaf(fk, pv[g].z, acc[f][4 * g + 2]);
          acc[f][4 * g + 3] = fmaf(fk, pv[g].w, acc[f][4 * g + 3]);
        }
      }
    }
#pragma unroll
    for (int f = 0; f < HEAD_FR; ++f)
#pragma unroll
      for (int g = 0; g < 4; ++g)
        reinterpret_cast<float4*>(s_part + (static_cast<size_t>(warp) * HEAD_FR + f) * E)[g * 32 + lane] =
            make_float4(acc[f][4 * g], acc[f][4 * g + 1], acc[f][4 * g + 2], acc[f][4 * g + 3]);
  }
  __syncthreads();
  for (int f = 0; f < HEAD_FR; ++f) {
#pragma unroll
    for (int j = 0; j < E / 256; ++j) {
      const int col = tid + j * 256;
      float yv = 0.f;
#pragma unroll
      for (int w8 = 0; w8 < 8; ++w8) yv += s_part[(static_cast<size_t>(w8) * HEAD_FR + f) * E + col];
      s_y[f][col] = yv;
      if (feat_out && f < nf) feat_out[static_cast<size_t>(b0 + f) * ld_feat + feat_col0 + col] = yv;
    }
  }
  clip_head_cosines<E>(s_y, s_red, s_inv, s_logit, b0, nf, text, n_text, group_off, n_groups, scale, reduce, logits,
                       reward, ld);
}

// The clip head from stored features: emb fp32 [n_frames, E], row b = frame b's un-normalised encode_image (what
// clip_head_kernel writes to feat_out). Same CTA shape, same thread -> column map and the same clip_head_cosines, so
// reward / logits are bit-identical to clip_head_kernel's on the frames the features came from. Memory-bound: E*4 bytes
// read per frame, no weights.
template <int E>
__global__ void __launch_bounds__(256)
clip_embedding_head_kernel(const float* __restrict__ emb, const float* __restrict__ text, int n_text,
                           const int* __restrict__ group_off, int n_groups, float scale, int reduce,
                           float* __restrict__ logits, float* __restrict__ reward, long long ld, long long n_frames) {
  static_assert(E % 256 == 0, "head widths must be multiples of the CTA size");
  __shared__ float s_y[HEAD_FR][E];
  __shared__ float s_red[8];
  __shared__ float s_inv[HEAD_FR];
  __shared__ float s_logit[HEAD_FR][HEAD_MAX_TEXT_TOTAL];
  const long long b0l = static_cast<long long>(blockIdx.x) * HEAD_FR;
  const int tid = threadIdx.x;
  const int nf = static_cast<int>(min(static_cast<long long>(HEAD_FR), n_frames - b0l));
  const float* src = emb + b0l * E;
  for (int f = 0; f < HEAD_FR; ++f)
#pragma unroll
    for (int j = 0; j < E / 256; ++j) {
      const int col = tid + j * 256;
      s_y[f][col] = f < nf ? __ldg(src + static_cast<size_t>(f) * E + col) : 0.f;
    }
  // reward / logits are addressed relative to b0: shift the bases so the shared code sees frame 0 at b0l
  clip_head_cosines<E>(s_y, s_red, s_inv, s_logit, 0, nf, text, n_text, group_off, n_groups, scale, reduce,
                       logits ? logits + b0l * n_text : nullptr, reward ? reward + b0l : nullptr, ld);
}

// Adapter gate + normalise + cosine. One CTA per frame, one warp per 512-wide scale (S warps).
//   feat, mlp fp32 [B, S*E]; text fp32 [n_text, S*E] (unit over S*E, or per-scale unit when ensemble), the rows of
//   n_groups groups at group_off as in clip_head_kernel; reward [n_groups, ld]
//   mlp == nullptr: `feat` already holds the gated feature a (what adapted_out receives; a stored embedding), and the
//   per-scale norms, dots and reductions below run on it unchanged, so relabeling it gives the frames path's bits.
template <int S, int E>
__global__ void __launch_bounds__(S * 32)
adapter_head_kernel(const float* __restrict__ feat, const float* __restrict__ mlp, float res,
                    const float* __restrict__ text, int n_text, const int* __restrict__ group_off, int n_groups,
                    float scale, int ensemble, int reduce, float* __restrict__ logits, float* __restrict__ reward,
                    long long ld, float* __restrict__ adapted_out) {
  __shared__ float s_n2[S];
  __shared__ float s_dot[S][HEAD_MAX_TEXT_TOTAL];
  const int b = blockIdx.x, sidx = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const size_t base = static_cast<size_t>(b) * S * E + static_cast<size_t>(sidx) * E;
  float a[E / 32];
  float n2 = 0.f;
#pragma unroll
  for (int i = 0; i < E / 32; ++i) {
    const int c = lane + i * 32;
    a[i] = mlp ? res * feat[base + c] + (1.0f - res) * mlp[base + c] : feat[base + c];
    n2 += a[i] * a[i];
    if (adapted_out) adapted_out[base + c] = a[i];
  }
  n2 = warp_sum(n2);
  if (lane == 0) s_n2[sidx] = n2;
  for (int t = 0; t < n_text; ++t) {
    const float* tr = text + static_cast<size_t>(t) * S * E + static_cast<size_t>(sidx) * E;
    float d = 0.f;
#pragma unroll
    for (int i = 0; i < E / 32; ++i) d = fmaf(a[i], __ldg(tr + lane + i * 32), d);
    d = warp_sum(d);
    if (lane == 0) s_dot[sidx][t] = d;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int g = 0; g < n_groups; ++g) {
      const int t0 = group_off[g], t1 = group_off[g + 1];
      const int n_use = reduce == REDUCE_MEAN ? t1 - t0 : 1;
      float racc = 0.f;
      for (int t = t0; t < t1; ++t) {
        float lg;
        if (ensemble) {
          float acc = 0.f;
          for (int s = 0; s < S; ++s) acc += s_dot[s][t] / fmaxf(sqrtf(s_n2[s]), 1e-12f);
          lg = scale * acc / static_cast<float>(S);
        } else {
          float tot = 0.f, d = 0.f;
          for (int s = 0; s < S; ++s) { tot += s_n2[s]; d += s_dot[s][t]; }
          lg = scale * (d / fmaxf(sqrtf(tot), 1e-12f));
        }
        if (logits) logits[static_cast<size_t>(b) * n_text + t] = lg;
        if (t - t0 < n_use) racc += lg;
      }
      if (reward) reward[g * ld + b] = racc / static_cast<float>(n_use);
    }
  }
}

// Goal-conditioned reward (label_reward.py:148-163,180-196): r_t = sign * || f_t - f_goal ||_2 where the
// goal is the LAST frame of the episode. One warp per frame. sign = -1 for "clip_goal_conditioned",
// +1 for the adapter "_goal_conditioned" variant (the reference omits the minus there, :193-195).
__global__ void __launch_bounds__(256)
goal_distance_kernel(const float* __restrict__ feat, int dim, const long long* __restrict__ frame_goal,
                     long long T, float sign, float* __restrict__ reward) {
  const long long t = static_cast<long long>(blockIdx.x) * 8 + (threadIdx.x >> 5);
  if (t >= T) return;
  const int lane = threadIdx.x & 31;
  const float* a = feat + t * dim;
  const float* g = feat + frame_goal[t] * dim;
  float s = 0.f;
  for (int k = lane; k < dim; k += 32) { const float d = a[k] - g[k]; s = fmaf(d, d, s); }
  s = warp_sum(s);
  if (lane == 0) reward[t] = sign * sqrtf(s);
}

}  // namespace arp
