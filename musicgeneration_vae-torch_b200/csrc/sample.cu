// sample.cu -- Bernoulli draw of every piano-roll cell from the decoder's logits, with a temperature.
//
// The decoder is trained with a per-cell BCE, so its output is a factorised Bernoulli distribution over the bar; the
// reference's sampling loop thresholds it at 0.3 (maker_bar.py:39).  This kernel draws from it instead:
//   p = 1 / (1 + expf(-(logit * inv_temperature))),  cell = (u < p),  u = (r >> 8) * 2^-24,
//   r = word (i % 4) of Philox4x32-10(counter = {i / 4, bar_index, song lo32, song hi32}, key = {seed lo32, seed hi32})
// with i the cell's index in its bar.  The random number is a function of (seed, song, bar, cell) alone, so a song
// does not depend on the batch it was sampled in.  p is the expression of fit_sigmoid_fwd_kernel (core.cu): at
// inv_temperature 1 it is bit-identical to the decoder's probability.  HBM bound: 4 B read + 4 B written per cell.
//
// bar_score_kernel scores a given roll under the same distribution: per bar, the negative log-likelihood in nats and
// the cell counts from which precision / recall / F1 follow.  HBM bound: 8 B read per cell.
#include "common.cuh"

namespace bvae {

constexpr int kBarCells = 96 * 60;              // 5760 = 720 groups of 8
constexpr int kGroupsPerBar = kBarCells / 8;

__device__ __forceinline__ float draw(float logit, float inv_t, uint32_t r) {
  const float p = prob_of_logit(logit * inv_t);
  const float u = (float)(r >> 8) * 5.9604644775390625e-8f;     // 2^-24: exact
  return u < p ? 1.f : 0.f;                                       // NaN p -> 0
}

// One thread per 8 consecutive cells of a bar: two float4 in, two Philox calls (counters 2j, 2j+1), two float4 out.
__global__ void __launch_bounds__(256) bernoulli_sample_kernel(const float* __restrict__ logits, int64_t groups,
                                                               float inv_t, uint2 key, int64_t song_base,
                                                               uint32_t bar_index, float* __restrict__ out) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t g = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; g < groups; g += stride) {
    const int64_t b = g / kGroupsPerBar;
    const uint32_t j = (uint32_t)(g - b * kGroupsPerBar);
    const uint64_t song = (uint64_t)(song_base + b);
    const uint32_t s_lo = (uint32_t)song, s_hi = (uint32_t)(song >> 32);
    const uint4 r0 = philox4x32_10(make_uint4(2 * j, bar_index, s_lo, s_hi), key);
    const uint4 r1 = philox4x32_10(make_uint4(2 * j + 1, bar_index, s_lo, s_hi), key);
    const float4 a = *reinterpret_cast<const float4*>(logits + g * 8);
    const float4 c = *reinterpret_cast<const float4*>(logits + g * 8 + 4);
    float4 o0, o1;
    o0.x = draw(a.x, inv_t, r0.x); o0.y = draw(a.y, inv_t, r0.y);
    o0.z = draw(a.z, inv_t, r0.z); o0.w = draw(a.w, inv_t, r0.w);
    o1.x = draw(c.x, inv_t, r1.x); o1.y = draw(c.y, inv_t, r1.y);
    o1.z = draw(c.z, inv_t, r1.z); o1.w = draw(c.w, inv_t, r1.w);
    *reinterpret_cast<float4*>(out + g * 8) = o0;
    *reinterpret_cast<float4*>(out + g * 8 + 4) = o1;
  }
}


// ---- the score of a given roll -----------------------------------------------------------------------------------
// One CTA per bar: 288 threads x 5 float4 of logits and 5 of targets = the 1440 float4 of a bar, no tail.  Each thread
// sums its 20 cells in a fixed order, the warps reduce by a fixed shuffle tree, thread 0 adds the 9 warp sums in warp
// order.  No atomics: a bar's result is a function of its logits and target alone (not of the grid, the bar count or
// the bar's row), so a chunked call gives the same bits as one call.
constexpr int kScoreThreads = 288;
constexpr int kScoreWarps = kScoreThreads / 32;
constexpr int kScoreVec = kBarCells / 4 / kScoreThreads;      // 5
static_assert(kScoreVec * 4 * kScoreThreads == kBarCells, "a bar must split evenly over the score CTA");

// softplus(x) = log(1 + e^x) in the stable form; +inf -> +inf, -inf -> 0, NaN -> NaN (through the log1pf term)
__device__ __forceinline__ float softplus_(float x) { return fmaxf(x, 0.f) + log1pf(expf(-fabsf(x))); }

struct BarScore {
  float nll;
  int tp, on, pos;
};

__device__ __forceinline__ void score_cell(float logit, float target, float inv_t, float threshold, BarScore& s) {
  const float l = logit * inv_t;
  const bool t = target != 0.f;
  const bool on = prob_of_logit(l) > threshold;      // NaN p is never on
  s.nll += softplus_(t ? -l : l);                     // -log p  or  -log(1 - p)
  s.tp += on && t;
  s.on += on;
  s.pos += t;
}

__global__ void __launch_bounds__(kScoreThreads) bar_score_kernel(const float* __restrict__ logits,
                                                                  const float* __restrict__ target, int64_t bars,
                                                                  float inv_t, float threshold,
                                                                  float* __restrict__ nll_out,
                                                                  int32_t* __restrict__ counts_out) {
  __shared__ BarScore part[kScoreWarps];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int64_t b = blockIdx.x; b < bars; b += gridDim.x) {
    const float4* lg = reinterpret_cast<const float4*>(logits + b * kBarCells) + threadIdx.x;
    const float4* tg = reinterpret_cast<const float4*>(target + b * kBarCells) + threadIdx.x;
    float4 l[kScoreVec], t[kScoreVec];
#pragma unroll
    for (int v = 0; v < kScoreVec; ++v) {
      l[v] = lg[v * kScoreThreads];
      t[v] = tg[v * kScoreThreads];
    }
    BarScore s = {0.f, 0, 0, 0};
#pragma unroll
    for (int v = 0; v < kScoreVec; ++v) {
      score_cell(l[v].x, t[v].x, inv_t, threshold, s);
      score_cell(l[v].y, t[v].y, inv_t, threshold, s);
      score_cell(l[v].z, t[v].z, inv_t, threshold, s);
      score_cell(l[v].w, t[v].w, inv_t, threshold, s);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      s.nll += __shfl_xor_sync(0xffffffffu, s.nll, o);
      s.tp += __shfl_xor_sync(0xffffffffu, s.tp, o);
      s.on += __shfl_xor_sync(0xffffffffu, s.on, o);
      s.pos += __shfl_xor_sync(0xffffffffu, s.pos, o);
    }
    if (lane == 0) part[warp] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
      BarScore r = part[0];
#pragma unroll
      for (int w = 1; w < kScoreWarps; ++w) {
        r.nll += part[w].nll;
        r.tp += part[w].tp;
        r.on += part[w].on;
        r.pos += part[w].pos;
      }
      nll_out[b] = r.nll;
      counts_out[3 * b] = r.tp;
      counts_out[3 * b + 1] = r.on;
      counts_out[3 * b + 2] = r.pos;
    }
    __syncthreads();                                  // part[] is rewritten by the next bar
  }
}

}  // namespace bvae

using namespace bvae;

extern "C" {

int bvae_bernoulli_sample(const float* logits, int64_t bars, float inv_temperature, uint64_t seed, int64_t song_base,
                          int32_t bar_index, float* out_f32, void* stream) {
  BVAE_REQUIRE(bars >= 0, BVAE_ERR_SHAPE, "bernoulli_sample: bars must be >= 0 (got %lld)", (long long)bars);
  BVAE_REQUIRE(isfinite(inv_temperature) && inv_temperature > 0.f, BVAE_ERR_SHAPE,
               "bernoulli_sample: inv_temperature must be finite and > 0 (got %g)", (double)inv_temperature);
  BVAE_REQUIRE((((uintptr_t)logits | (uintptr_t)out_f32) & 15) == 0, BVAE_ERR_ALIGN,
               "bernoulli_sample: logits and out_f32 must be 16-byte aligned");
  if (bars == 0) return BVAE_OK;
  const int64_t groups = bars * kGroupsPerBar;
  int64_t grid = ceil_div64(groups, 256);
  if (grid > 148 * 8) grid = 148 * 8;       // 8 resident 256-thread CTAs per SM, grid-stride beyond
  const uint2 key = make_uint2((uint32_t)seed, (uint32_t)(seed >> 32));
  bernoulli_sample_kernel<<<(int)grid, 256, 0, (cudaStream_t)stream>>>(logits, groups, inv_temperature, key, song_base,
                                                                       (uint32_t)bar_index, out_f32);
  return check_launch("bernoulli_sample");
}

int bvae_bar_score(const float* logits, const float* target, int64_t bars, float inv_temperature, float threshold,
                   float* nll_out, int32_t* counts_out, void* stream) {
  BVAE_REQUIRE(bars >= 0, BVAE_ERR_SHAPE, "bar_score: bars must be >= 0 (got %lld)", (long long)bars);
  BVAE_REQUIRE(isfinite(inv_temperature) && inv_temperature > 0.f, BVAE_ERR_SHAPE,
               "bar_score: inv_temperature must be finite and > 0 (got %g)", (double)inv_temperature);
  BVAE_REQUIRE(isfinite(threshold), BVAE_ERR_SHAPE, "bar_score: threshold must be finite (got %g)", (double)threshold);
  BVAE_REQUIRE((((uintptr_t)logits | (uintptr_t)target) & 15) == 0, BVAE_ERR_ALIGN,
               "bar_score: logits and target must be 16-byte aligned");
  BVAE_REQUIRE((((uintptr_t)nll_out | (uintptr_t)counts_out) & 3) == 0, BVAE_ERR_ALIGN,
               "bar_score: nll_out and counts_out must be 4-byte aligned");
  if (bars == 0) return BVAE_OK;
  const int64_t grid = bars < 148 * 16 ? bars : 148 * 16;      // bar-stride beyond
  bar_score_kernel<<<(int)grid, kScoreThreads, 0, (cudaStream_t)stream>>>(logits, target, bars, inv_temperature,
                                                                          threshold, nll_out, counts_out);
  return check_launch("bar_score");
}

}  // extern "C"
