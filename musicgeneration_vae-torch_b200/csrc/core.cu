// core.cu -- library state (errors, launch counter) and the small memory-bound kernels:
// weight packing, column sums, fit2+sigmoid, BCE, reparameterise+KL, flat Adam.
#include <stdarg.h>
#include <stdlib.h>
#include <atomic>
#include "common.cuh"
#include <vector>
#include <mutex>
#include <string>
#include <unordered_map>

namespace bvae {

static thread_local char g_err[1024] = "";
static std::atomic<uint64_t> g_launches{0};

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}
static thread_local char g_kernel[160] = "";
static std::atomic<int> g_det{-1};

void note_kernel(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_kernel, sizeof(g_kernel), fmt, ap);
  va_end(ap);
}
bool deterministic() {
  int v = g_det.load(std::memory_order_relaxed);
  if (v < 0) {
    const char* e = getenv("BVAE_DETERMINISTIC");
    v = (e && e[0] == '1') ? 1 : 0;
    g_det.store(v, std::memory_order_relaxed);
  }
  return v == 1;
}
// kernel-variant switches: bvae_set_option overrides, else the environment variable of the same name, else the default
static std::mutex g_opt_mu;
static std::unordered_map<std::string, int> g_opts;
int option(const char* name, int dflt) {
  {
    std::lock_guard<std::mutex> g(g_opt_mu);
    auto it = g_opts.find(name);
    if (it != g_opts.end()) return it->second;
  }
  const char* e = getenv(name);
  return (e && e[0]) ? atoi(e) : dflt;
}
void count_launch(int n) { g_launches.fetch_add((uint64_t)n, std::memory_order_relaxed); }
int check_launch(const char* what) {
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) {
    set_error("%s: %s", what, cudaGetErrorString(e));
    return BVAE_ERR_CUDA;
  }
  count_launch(1);
  return BVAE_OK;
}

// ---------------------------------------------------------------------------------------------------
// weight packing: fp32 parameter (reference layout) -> bf16 GEMM operand rows
// ---------------------------------------------------------------------------------------------------
struct PackPerm {
  int32_t p[BVAE_MAX_TAPS];
};

__global__ void pack_weight_kernel(const float* __restrict__ src, bf16* __restrict__ dst, int R, int T, int Cc,
                                   int64_t sr, int64_t sc, PackPerm perm, int dst_pitch) {
  // one thread per destination element; destination is contiguous along c so writes coalesce, reads are a gather
  const int64_t total = (int64_t)R * T * Cc;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int c = (int)(i % Cc);
    const int tp = (int)((i / Cc) % T);
    const int r = (int)(i / ((int64_t)Cc * T));
    dst[(int64_t)r * dst_pitch + (int64_t)tp * Cc + c] = f2bf(src[r * sr + c * sc + perm.p[tp]]);
  }
}

// Batched repack: one CTA per (8 rows x 64 columns x all taps) tile of one job.  The tile is read in the order that is
// contiguous in the SOURCE (taps fastest, then whichever of r / c has the smaller stride), staged in shared memory
// and written as 128-byte destination rows.
struct PackJobDev {
  const float* src;
  bf16* dst;
  int R, T, Cc, dst_pitch;
  long long sr, sc;
  int perm[BVAE_MAX_TAPS];
  int block0, ctiles;
};

__global__ void __launch_bounds__(256) pack_batch_kernel(const PackJobDev* __restrict__ jobs, int njobs) {
  constexpr int RT = 8, CT = 64, LD = CT + 2;
  __shared__ PackJobDev j;
  __shared__ __align__(16) bf16 tile[RT * BVAE_MAX_TAPS * LD];
  __shared__ int jsel;
  if (threadIdx.x == 0) {
    int lo = 0, hi = njobs - 1;
    while (lo < hi) {
      const int mid = (lo + hi + 1) >> 1;
      if (jobs[mid].block0 <= (int)blockIdx.x) lo = mid; else hi = mid - 1;
    }
    jsel = lo;
  }
  __syncthreads();
  if (threadIdx.x < sizeof(PackJobDev) / 4)
    reinterpret_cast<int*>(&j)[threadIdx.x] = reinterpret_cast<const int*>(jobs + jsel)[threadIdx.x];
  __syncthreads();
  const int local = blockIdx.x - j.block0;
  const int r0 = (local / j.ctiles) * RT, c0 = (local % j.ctiles) * CT;
  const int nr = min(RT, j.R - r0), nc = min(CT, j.Cc - c0), T = j.T;
  const float* src = j.src + r0 * j.sr + c0 * j.sc;
  // every thread owns (row, column) pairs and walks their T taps (T consecutive floats): no integer divisions, and a
  // warp covers a contiguous run of the source in whichever of r / c is the faster source dimension
#pragma unroll
  for (int k = 0; k < RT * CT / 256; ++k) {
    const int e = threadIdx.x + 256 * k;
    const int r = (j.sr <= j.sc) ? (e & (RT - 1)) : (e / CT);
    const int c = (j.sr <= j.sc) ? (e / RT) : (e & (CT - 1));
    if (r < nr && c < nc) {
      const float* sp = src + r * j.sr + c * j.sc;
      bf16* tp_ = tile + (r * T) * LD + c;
      for (int tp = 0; tp < T; ++tp) tp_[tp * LD] = f2bf(sp[j.perm[tp]]);
    }
  }
  __syncthreads();
  const int rr = threadIdx.x >> 5, c2 = threadIdx.x & 31;        // warp = tile row r, lane = channel pair
  if (rr < nr) {
    bf16* drow = j.dst + (int64_t)(r0 + rr) * j.dst_pitch + c0;
    if (nc == CT && (j.Cc & 1) == 0 && (j.dst_pitch & 1) == 0) {
      for (int tp = 0; tp < T; ++tp)
        *reinterpret_cast<uint32_t*>(drow + (int64_t)tp * j.Cc + 2 * c2) =
            *reinterpret_cast<const uint32_t*>(tile + (rr * T + tp) * LD + 2 * c2);
    } else {
      for (int tp = 0; tp < T; ++tp)
        for (int c = c2; c < nc; c += 32) drow[(int64_t)tp * j.Cc + c] = tile[(rr * T + tp) * LD + c];
    }
  }
}

// ---------------------------------------------------------------------------------------------------
// column sums (bias gradients)
// ---------------------------------------------------------------------------------------------------
template <typename T>
__global__ void colsum_kernel(const T* __restrict__ x, int64_t rows, int C, int pitch, float* __restrict__ out,
                              int rows_per_block) {
  __shared__ float red[8][33];
  const int c = blockIdx.x * 32 + threadIdx.x;
  const int64_t r0 = (int64_t)blockIdx.y * rows_per_block;
  const int64_t r1 = min(rows, r0 + rows_per_block);
  float acc = 0.f;
  if (c < C)
    for (int64_t r = r0 + threadIdx.y; r < r1; r += 8) acc += (float)x[r * pitch + c];
  red[threadIdx.y][threadIdx.x] = acc;
  __syncthreads();
  if (threadIdx.y == 0 && c < C) {
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) s += red[i][threadIdx.x];
    atomicAdd(out + c, s);
  }
}

// ---------------------------------------------------------------------------------------------------
// fit2 (C -> 1) + sigmoid ; BCE ; fused backward
// rows are pixels; G = C/8 lanes cooperate on one row (16-byte loads).
// ---------------------------------------------------------------------------------------------------
__global__ void fit_sigmoid_fwd_kernel(const bf16* __restrict__ x, int x_pitch, const float* __restrict__ w,
                                       int64_t rows, int C, float* __restrict__ logits, float* __restrict__ recon) {
  const int G = C / 8;  // lanes per row (power of two <= 32)
  const int lane = threadIdx.x & 31;
  const int sub = lane % G;
  const int64_t rows_per_warp = 32 / G;
  const int64_t warp = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
  const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  float wv[8];
  ldg8f(w + sub * 8, wv);
  for (int64_t base = warp * rows_per_warp; base < rows; base += nwarps * rows_per_warp) {
    const int64_t row = base + lane / G;
    float acc = 0.f;
    if (row < rows) {
      float xv[8];
      unpack8(ldg8(x + row * x_pitch + sub * 8), xv);
#pragma unroll
      for (int i = 0; i < 8; ++i) acc += xv[i] * wv[i];
    }
    for (int o = G >> 1; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if (sub == 0 && row < rows) {
      if (logits) logits[row] = acc;
      recon[row] = prob_of_logit(acc);
    }
  }
}

__constant__ float c_pitch_prior[60] = {
    0.0079033f,  0.00712255f, 0.01189558f, 0.00953322f, 0.01102056f, 0.01156428f, 0.01136433f, 0.01637716f,
    0.01211462f, 0.01776168f, 0.01644157f, 0.0171948f,  0.01922302f, 0.01582762f, 0.02385192f, 0.02001634f,
    0.02312213f, 0.02348127f, 0.02263083f, 0.0268141f,  0.02373071f, 0.02942328f, 0.0272045f,  0.0304963f,
    0.03032582f, 0.02782333f, 0.03458292f, 0.03230801f, 0.03388906f, 0.03283811f, 0.03093611f, 0.03616363f,
    0.03006419f, 0.03296618f, 0.02867032f, 0.02654072f, 0.02609579f, 0.01954488f, 0.02251165f, 0.01813882f,
    0.01599178f, 0.01313839f, 0.01104167f, 0.01169814f, 0.00756204f, 0.00793332f, 0.00601032f, 0.00540243f,
    0.00512497f, 0.00286655f, 0.00308927f, 0.00260029f, 0.00184589f, 0.00166959f, 0.00103728f, 0.00112497f,
    0.00071164f, 0.00052543f, 0.00072274f, 0.00038808f};

__device__ __forceinline__ float smooth_target(float t, int64_t row, int smoothing) {
  if (!smoothing) return t;
  // graph/loss/bar_loss.py:28: labels*0.82 + 0.1/60 + prior*0.08, prior broadcast over the pitch (last) axis
  return t * 0.82f + (0.1f / 60.f) + c_pitch_prior[row % 60] * 0.08f;
}

__global__ void bce_fwd_kernel(const float* __restrict__ recon, const float* __restrict__ target, int64_t rows,
                               int smoothing, float inv_rows, float* __restrict__ loss_out) {
  float lsum = 0.f, miss = 0.f;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < rows; i += (int64_t)gridDim.x * blockDim.x) {
    const float p = recon[i];
    const float t = target[i];
    const float ts = smooth_target(t, i, smoothing);
    const float lp = fmaxf(logf(p), -100.f);          // nn.BCELoss clamps each log term at -100
    const float l1p = fmaxf(logf(1.f - p), -100.f);
    lsum -= ts * lp + (1.f - ts) * l1p;
    const float o = p > 0.3f ? 1.f : 0.f;             // bar_loss.py:31-32
    miss += (t - o > 0.0001f) ? 1.f : 0.f;
  }
  __shared__ float s0[32], s1[32];
  lsum = warp_sum(lsum);
  miss = warp_sum(miss);
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  if (lane == 0) { s0[wid] = lsum; s1[wid] = miss; }
  __syncthreads();
  if (wid == 0) {
    const int nw = blockDim.x >> 5;
    float a = lane < nw ? s0[lane] : 0.f, b = lane < nw ? s1[lane] : 0.f;
    a = warp_sum(a);
    b = warp_sum(b);
    if (lane == 0) {
      atomicAdd(loss_out, a * inv_rows);
      atomicAdd(loss_out + 1, b);
    }
  }
}

__global__ void bce_bwd_kernel(const float* __restrict__ recon, const float* __restrict__ target, int64_t rows,
                               int smoothing, float gscale, float* __restrict__ drecon) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < rows; i += (int64_t)gridDim.x * blockDim.x) {
    const float p = recon[i];
    const float ts = smooth_target(target[i], i, smoothing);
    drecon[i] = gscale * (p - ts) / fmaxf(p * (1.f - p), 1e-12f);
  }
}

__global__ void fit_sigmoid_bce_bwd_kernel(const bf16* __restrict__ x, int x_pitch, const float* __restrict__ w,
                                           const float* __restrict__ recon, const float* __restrict__ target,
                                           const float* __restrict__ drecon, float gscale, int smoothing,
                                           int64_t rows, int C, bf16* __restrict__ dx, int dx_pitch,
                                           float* __restrict__ dw) {
  const int G = C / 8;
  const int lane = threadIdx.x & 31;
  const int sub = lane % G;
  const int64_t rows_per_warp = 32 / G;
  const int64_t warp = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
  const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  float wv[8], dwv[8];
  ldg8f(w + sub * 8, wv);
#pragma unroll
  for (int i = 0; i < 8; ++i) dwv[i] = 0.f;
  for (int64_t base = warp * rows_per_warp; base < rows; base += nwarps * rows_per_warp) {
    const int64_t row = base + lane / G;
    if (row < rows) {
      const float p = recon[row];
      const float pq = p * (1.f - p);
      float g;
      if (drecon) {
        g = drecon[row] * pq;
      } else {
        const float ts = smooth_target(target[row], row, smoothing);
        g = gscale * (p - ts) / fmaxf(pq, 1e-12f) * pq;   // BCELoss backward (eps 1e-12) then sigmoid backward
      }
      float xv[8], dv[8];
      unpack8(ldg8(x + row * x_pitch + sub * 8), xv);
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        dwv[i] += g * xv[i];
        dv[i] = g * wv[i];
      }
      stg8(dx + row * dx_pitch + sub * 8, pack8(dv));
    }
  }
  // reduce dw over the rows of this warp (lanes with equal sub), then over the block, then one atomic per channel
  for (int o = G; o < 32; o <<= 1)
#pragma unroll
    for (int i = 0; i < 8; ++i) dwv[i] += __shfl_xor_sync(0xffffffffu, dwv[i], o);
  __shared__ float sdw[256];
  for (int i = threadIdx.x; i < C; i += blockDim.x) sdw[i] = 0.f;
  __syncthreads();
  if (lane < G)
#pragma unroll
    for (int i = 0; i < 8; ++i) atomicAdd(&sdw[sub * 8 + i], dwv[i]);
  __syncthreads();
  for (int i = threadIdx.x; i < C; i += blockDim.x) atomicAdd(dw + i, sdw[i]);
}

// ---------------------------------------------------------------------------------------------------
// reparameterise + KL
// ---------------------------------------------------------------------------------------------------
__global__ void reparam_kl_fwd_kernel(const float* __restrict__ mu, const float* __restrict__ lv,
                                      const float* __restrict__ eps, float* __restrict__ z, float* __restrict__ kl,
                                      int64_t n) {
  float acc = 0.f;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const float m = mu[i], l = lv[i];
    z[i] = m + eps[i] * expf(0.5f * l);
    acc += 1.f + l - m * m - expf(l);
  }
  __shared__ float s[32];
  acc = warp_sum(acc);
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  if (lane == 0) s[wid] = acc;
  __syncthreads();
  if (wid == 0) {
    float a = lane < (blockDim.x >> 5) ? s[lane] : 0.f;
    a = warp_sum(a);
    if (lane == 0) atomicAdd(kl, -0.5f * a);
  }
}

__global__ void reparam_kl_bwd_kernel(const float* __restrict__ mu, const float* __restrict__ lv,
                                      const float* __restrict__ eps, const float* __restrict__ dz, float gkl,
                                      float* __restrict__ dmu, float* __restrict__ dlv, int64_t n) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const float m = mu[i], l = lv[i], g = dz ? dz[i] : 0.f;
    dmu[i] = g + gkl * m;
    dlv[i] = g * eps[i] * 0.5f * expf(0.5f * l) + gkl * 0.5f * (expf(l) - 1.f);
  }
}

// ---------------------------------------------------------------------------------------------------
// flat Adam: p, g, m, v are one contiguous fp32 bucket each (all generator parameters)
// 16 B/param read + 12 B/param written
// ---------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) adam_kernel(float* __restrict__ p, const float* __restrict__ g,
                                                   float* __restrict__ m, float* __restrict__ v, int64_t n4,
                                                   int64_t n, float b1, float b2, float eps, float step_size,
                                                   float inv_sqrt_bc2, float gscale, const float* __restrict__ hyp) {
  if (hyp) {      // step-dependent scalars from device memory: lets a captured CUDA graph replay the launch unchanged
    step_size = hyp[0]; inv_sqrt_bc2 = hyp[1]; b1 = hyp[2]; b2 = hyp[3]; eps = hyp[4]; gscale = hyp[5];
  }
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n4; i += stride) {
    float4 pp = reinterpret_cast<float4*>(p)[i];
    float4 gg = reinterpret_cast<const float4*>(g)[i];
    float4 mm = reinterpret_cast<float4*>(m)[i];
    float4 vv = reinterpret_cast<float4*>(v)[i];
    float* pa = &pp.x; float* ga = &gg.x; float* ma = &mm.x; float* va = &vv.x;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const float gk = ga[k] * gscale;
      ma[k] = b1 * ma[k] + (1.f - b1) * gk;
      va[k] = b2 * va[k] + (1.f - b2) * gk * gk;
      pa[k] -= step_size * ma[k] / (sqrtf(va[k]) * inv_sqrt_bc2 + eps);
    }
    reinterpret_cast<float4*>(p)[i] = pp;
    reinterpret_cast<float4*>(m)[i] = mm;
    reinterpret_cast<float4*>(v)[i] = vv;
  }
  // tail (n not a multiple of 4)
  for (int64_t i = n4 * 4 + blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += stride) {
    const float gk = g[i] * gscale;
    const float mk = b1 * m[i] + (1.f - b1) * gk;
    const float vk = b2 * v[i] + (1.f - b2) * gk * gk;
    m[i] = mk; v[i] = vk;
    p[i] -= step_size * mk / (sqrtf(vk) * inv_sqrt_bc2 + eps);
  }
}

__global__ void cast_f32_bf16_kernel(const float* __restrict__ s, bf16* __restrict__ d, int64_t n) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    d[i] = f2bf(s[i]);
}

}  // namespace bvae

using namespace bvae;

extern "C" {

int bvae_version(void) { return 100; }
const char* bvae_last_error(void) { return bvae::g_err; }
uint64_t bvae_launch_count(void) { return bvae::g_launches.load(); }
void bvae_launch_count_reset(void) { bvae::g_launches.store(0); }
void bvae_launch_count_add(uint64_t n) { bvae::g_launches.fetch_add(n); }
const char* bvae_last_kernel(void) { return bvae::g_kernel; }
void bvae_set_deterministic(int on) { bvae::g_det.store(on ? 1 : 0); }
void bvae_set_option(const char* name, int value) {
  std::lock_guard<std::mutex> g(bvae::g_opt_mu);
  if (value < 0) bvae::g_opts.erase(name);
  else bvae::g_opts[name] = value;
}
int bvae_get_option(const char* name, int dflt) { return bvae::option(name, dflt); }
int bvae_deterministic(void) { return bvae::deterministic() ? 1 : 0; }

int bvae_device_ok(void) {
  int dev = 0;
  cudaDeviceProp prop;
  if (cudaGetDevice(&dev) != cudaSuccess || cudaGetDeviceProperties(&prop, dev) != cudaSuccess) {
    set_error("no CUDA device");
    return 0;
  }
  if (prop.major != 10) {
    set_error("libbarvae is built for sm_100a only; device is sm_%d%d", prop.major, prop.minor);
    return 0;
  }
  return 1;
}

static inline int grid_for(int64_t n, int block, int max_blocks = 148 * 8) {
  int64_t g = (n + block - 1) / block;
  if (g < 1) g = 1;
  if (g > max_blocks) g = max_blocks;
  return (int)g;
}

int bvae_pack_weight(const float* src, void* dst, int R, int T, int Cc, int64_t sr, int64_t sc,
                     const int32_t* perm, int dst_pitch, void* stream) {
  BVAE_REQUIRE(T >= 1 && T <= BVAE_MAX_TAPS, BVAE_ERR_SHAPE, "pack_weight: T=%d out of range", T);
  BVAE_REQUIRE(dst_pitch >= T * Cc, BVAE_ERR_SHAPE, "pack_weight: dst_pitch too small");
  PackPerm pp;
  for (int i = 0; i < T; ++i) pp.p[i] = perm ? perm[i] : i;
  const int64_t total = (int64_t)R * T * Cc;
  pack_weight_kernel<<<grid_for(total, 256), 256, 0, (cudaStream_t)stream>>>(src, (bf16*)dst, R, T, Cc, sr, sc, pp,
                                                                              dst_pitch);
  return check_launch("pack_weight");
}

struct bvae_pack_plan {
  bvae::PackJobDev* jobs;
  int njobs, nblocks;
};

int bvae_pack_plan_create(const bvae_pack_job* jobs, int njobs, bvae_pack_plan** out) {
  BVAE_REQUIRE(jobs && out && njobs > 0, BVAE_ERR_SHAPE, "pack_plan: no jobs");
  std::vector<bvae::PackJobDev> host((size_t)njobs);
  long long blocks = 0;
  for (int i = 0; i < njobs; ++i) {
    const bvae_pack_job& a = jobs[i];
    BVAE_REQUIRE(a.T >= 1 && a.T <= BVAE_MAX_TAPS, BVAE_ERR_SHAPE, "pack_plan: job %d: T=%d out of range", i, a.T);
    BVAE_REQUIRE(a.R > 0 && a.Cc > 0 && a.dst_pitch >= a.T * a.Cc, BVAE_ERR_SHAPE, "pack_plan: job %d: bad shape", i);
    BVAE_REQUIRE(a.src && a.dst, BVAE_ERR_SHAPE, "pack_plan: job %d: null pointer", i);
    bvae::PackJobDev& d = host[(size_t)i];
    d.src = a.src; d.dst = (bf16*)a.dst;
    d.R = a.R; d.T = a.T; d.Cc = a.Cc; d.dst_pitch = a.dst_pitch; d.sr = a.sr; d.sc = a.sc;
    for (int t = 0; t < BVAE_MAX_TAPS; ++t) d.perm[t] = t < a.T ? a.perm[t] : 0;
    d.block0 = (int)blocks;
    d.ctiles = ceil_div(a.Cc, 64);
    blocks += (long long)ceil_div(a.R, 8) * d.ctiles;
    BVAE_REQUIRE(blocks < (1ll << 31), BVAE_ERR_SHAPE, "pack_plan: too many tiles");
  }
  bvae_pack_plan* pl = new bvae_pack_plan;
  pl->njobs = njobs; pl->nblocks = (int)blocks; pl->jobs = nullptr;
  cudaError_t e = cudaMalloc(&pl->jobs, sizeof(bvae::PackJobDev) * (size_t)njobs);
  if (e == cudaSuccess) e = cudaMemcpy(pl->jobs, host.data(), sizeof(bvae::PackJobDev) * (size_t)njobs, cudaMemcpyHostToDevice);
  if (e != cudaSuccess) {
    if (pl->jobs) cudaFree(pl->jobs);
    delete pl;
    BVAE_REQUIRE(false, BVAE_ERR_CUDA, "pack_plan: %s", cudaGetErrorString(e));
  }
  *out = pl;
  return 0;
}

int bvae_pack_plan_run(const bvae_pack_plan* plan, void* stream) {
  BVAE_REQUIRE(plan && plan->jobs, BVAE_ERR_SHAPE, "pack_plan_run: null plan");
  bvae::pack_batch_kernel<<<plan->nblocks, 256, 0, (cudaStream_t)stream>>>(plan->jobs, plan->njobs);
  return check_launch("pack_batch");
}

void bvae_pack_plan_destroy(bvae_pack_plan* plan) {
  if (!plan) return;
  if (plan->jobs) cudaFree(plan->jobs);
  delete plan;
}

int bvae_colsum(const void* x, int x_f32, int64_t rows, int C, int pitch, float* out, void* stream) {
  BVAE_REQUIRE(rows > 0 && C > 0, BVAE_ERR_SHAPE, "colsum: empty");
  int rpb = (int)ceil_div64(rows, 148 * 4);
  if (rpb < 64) rpb = 64;
  dim3 grid(ceil_div(C, 32), (unsigned)ceil_div64(rows, rpb));
  dim3 block(32, 8);
  if (x_f32)
    colsum_kernel<float><<<grid, block, 0, (cudaStream_t)stream>>>((const float*)x, rows, C, pitch, out, rpb);
  else
    colsum_kernel<bf16><<<grid, block, 0, (cudaStream_t)stream>>>((const bf16*)x, rows, C, pitch, out, rpb);
  return check_launch("colsum");
}

static int check_fit_C(int C) { return C >= 8 && C <= 256 && (C & (C - 1)) == 0; }

int bvae_fit_sigmoid_fwd(const void* x, int x_pitch, const float* w, int64_t rows, int C, float* logits,
                         float* recon, void* stream) {
  BVAE_REQUIRE(check_fit_C(C), BVAE_ERR_SHAPE, "fit_sigmoid: C=%d must be a power of two in [8,256]", C);
  BVAE_REQUIRE(x_pitch % 8 == 0, BVAE_ERR_ALIGN, "fit_sigmoid: pitch must be a multiple of 8");
  const int64_t warps = ceil_div64(rows, 32 / (C / 8));
  fit_sigmoid_fwd_kernel<<<grid_for(warps * 32, 256, 148 * 16), 256, 0, (cudaStream_t)stream>>>(
      (const bf16*)x, x_pitch, w, rows, C, logits, recon);
  return check_launch("fit_sigmoid_fwd");
}

int bvae_bce_fwd(const float* recon, const float* target, int64_t rows, int smoothing, float* loss_out,
                 void* stream) {
  // deterministic mode: one CTA, so the two scalars are reduced in a fixed order (no float atomics across CTAs)
  bce_fwd_kernel<<<deterministic() ? 1 : grid_for(rows, 256, 148 * 4), 256, 0, (cudaStream_t)stream>>>(recon, target, rows, smoothing,
                                                                                1.f / (float)rows, loss_out);
  return check_launch("bce_fwd");
}

int bvae_bce_bwd(const float* recon, const float* target, int64_t rows, int smoothing, float gscale, float* drecon,
                 void* stream) {
  bce_bwd_kernel<<<grid_for(rows, 256, 148 * 4), 256, 0, (cudaStream_t)stream>>>(recon, target, rows, smoothing,
                                                                                gscale, drecon);
  return check_launch("bce_bwd");
}

int bvae_fit_sigmoid_bce_bwd(const void* x, int x_pitch, const float* w, const float* recon, const float* target,
                             const float* drecon, float gscale, int smoothing, int64_t rows, int C, void* dx,
                             int dx_pitch, float* dw, void* stream) {
  BVAE_REQUIRE(check_fit_C(C), BVAE_ERR_SHAPE, "fit_sigmoid_bwd: C=%d must be a power of two in [8,256]", C);
  BVAE_REQUIRE(x_pitch % 8 == 0 && dx_pitch % 8 == 0, BVAE_ERR_ALIGN, "fit_sigmoid_bwd: pitch % 8 != 0");
  const int64_t warps = ceil_div64(rows, 32 / (C / 8));
  fit_sigmoid_bce_bwd_kernel<<<grid_for(warps * 32, 256, 148 * 4), 256, 0, (cudaStream_t)stream>>>(
      (const bf16*)x, x_pitch, w, recon, target, drecon, gscale, smoothing, rows, C, (bf16*)dx, dx_pitch, dw);
  return check_launch("fit_sigmoid_bce_bwd");
}

int bvae_reparam_kl_fwd(const float* mu, const float* logvar, const float* eps, float* z, float* kl_out, int64_t n,
                        void* stream) {
  reparam_kl_fwd_kernel<<<grid_for(n, 256, 148 * 4), 256, 0, (cudaStream_t)stream>>>(mu, logvar, eps, z, kl_out, n);
  return check_launch("reparam_kl_fwd");
}

int bvae_reparam_kl_bwd(const float* mu, const float* logvar, const float* eps, const float* dz, float gkl,
                        float* dmu, float* dlogvar, int64_t n, void* stream) {
  reparam_kl_bwd_kernel<<<grid_for(n, 256, 148 * 4), 256, 0, (cudaStream_t)stream>>>(mu, logvar, eps, dz, gkl, dmu,
                                                                                    dlogvar, n);
  return check_launch("reparam_kl_bwd");
}

int bvae_adam_step(float* p, const float* g, float* m, float* v, int64_t n, float lr, float b1, float b2, float eps,
                   int step, float grad_scale, void* stream) {
  BVAE_REQUIRE(step >= 1, BVAE_ERR_SHAPE, "adam: step must be >= 1");
  BVAE_REQUIRE((((uintptr_t)p | (uintptr_t)g | (uintptr_t)m | (uintptr_t)v) & 15) == 0, BVAE_ERR_ALIGN,
               "adam: buffers must be 16-byte aligned");
  const double bc1 = 1.0 - pow((double)b1, step), bc2 = 1.0 - pow((double)b2, step);
  const float step_size = (float)(lr / bc1);
  const float inv_sqrt_bc2 = (float)(1.0 / sqrt(bc2));
  const int64_t n4 = n / 4;
  adam_kernel<<<148 * 8, 256, 0, (cudaStream_t)stream>>>(p, g, m, v, n4, n, b1, b2, eps, step_size, inv_sqrt_bc2,
                                                        grad_scale, nullptr);
  return check_launch("adam");
}

void bvae_adam_hyper(float lr, float b1, float b2, float eps, int step, float grad_scale, float* out6);
}  // extern "C" (reopened below: a kernel cannot have C linkage)
__global__ void adam_hyper_kernel(float* out, float a, float b, float c, float d, float e, float f) {
  out[0] = a; out[1] = b; out[2] = c; out[3] = d; out[4] = e; out[5] = f;
}
extern "C" {

int bvae_adam_hyper_upload(float lr, float b1, float b2, float eps, int step, float grad_scale, float* hyper_dev,
                           void* stream) {
  BVAE_REQUIRE(step >= 1 && hyper_dev, BVAE_ERR_SHAPE, "adam_hyper_upload: step must be >= 1, hyper_dev non-NULL");
  float h[6];
  bvae_adam_hyper(lr, b1, b2, eps, step, grad_scale, h);
  adam_hyper_kernel<<<1, 1, 0, (cudaStream_t)stream>>>(hyper_dev, h[0], h[1], h[2], h[3], h[4], h[5]);
  return check_launch("adam_hyper");
}

void bvae_adam_hyper(float lr, float b1, float b2, float eps, int step, float grad_scale, float* out6) {
  const double bc1 = 1.0 - pow((double)b1, step), bc2 = 1.0 - pow((double)b2, step);
  out6[0] = (float)(lr / bc1);
  out6[1] = (float)(1.0 / sqrt(bc2));
  out6[2] = b1; out6[3] = b2; out6[4] = eps; out6[5] = grad_scale;
}

int bvae_adam_step_dev(float* p, const float* g, float* m, float* v, int64_t n, const float* hyper_dev, void* stream) {
  BVAE_REQUIRE(hyper_dev != nullptr, BVAE_ERR_SHAPE, "adam_dev: hyper_dev is NULL");
  BVAE_REQUIRE((((uintptr_t)p | (uintptr_t)g | (uintptr_t)m | (uintptr_t)v) & 15) == 0, BVAE_ERR_ALIGN,
               "adam: buffers must be 16-byte aligned");
  adam_kernel<<<148 * 8, 256, 0, (cudaStream_t)stream>>>(p, g, m, v, n / 4, n, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, hyper_dev);
  return check_launch("adam");
}

int bvae_f32_to_bf16(const float* src, void* dst, int64_t n, void* stream) {
  cast_f32_bf16_kernel<<<grid_for(n, 256), 256, 0, (cudaStream_t)stream>>>(src, (bf16*)dst, n);
  return check_launch("f32_to_bf16");
}

}  // extern "C"
