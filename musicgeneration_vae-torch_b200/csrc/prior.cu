// prior.cu -- fp64 first and second moments of a set of latents, for the Gaussian prior fitted to the encoder's
// output (prior.py).
//
//   sum[j]     += sum_i z[i][j]
//   gram[j][k] += sum_i z[i][j] * z[i][k]        (k >= j only: the lower triangle is neither read nor written)
//
// Order contract: every output element starts from the value already in memory and adds its rows one at a time in
// increasing row order, each product formed in fp64.  A product of two fp32 values is exact in fp64, so
// fma(a, b, acc) == acc + a*b bit for bit and the compiler's DFMA changes nothing.  No atomics, no split of the row
// range across CTAs, no DMMA (whose internal summation order is unspecified): consecutive calls over consecutive
// chunks of rows give the same bits as one call over all of them.
//
// Grid: one CTA per upper-triangular kTile x kTile tile of gram (666 tiles for d = 1152, which balances 148 SMs better
// than the 171 tiles of 64-wide ones).  Each CTA streams all n rows in slabs of kSlab rows: the slab's two column blocks
// are loaded as fp32 (coalesced, one column per thread, prefetched into registers while the previous slab is used),
// converted to fp64 once into shared memory, and every thread accumulates a 4 x 4 fp64 register tile.  The sum comes
// from the diagonal tiles' first warp.  An 8192-latent chunk (38 MB) is read from L2 after the first wave of tiles.
#include "common.cuh"

namespace bvae {

constexpr int kTile = 32;                          // gram tile edge
constexpr int kSlab = 32;                          // rows staged per shared-memory slab
constexpr int kMomThreads = 64;                    // 8 x 8 threads, 4 x 4 outputs each
constexpr int kSub = kTile / 8;                    // 4
static_assert(kMomThreads == 2 * kTile, "one thread per staged column (two column blocks)");

__global__ void __launch_bounds__(kMomThreads, 8)
latent_moments_kernel(const float* __restrict__ z, int64_t n, int d, int64_t ld, int nb, double* __restrict__ sum,
                      double* __restrict__ gram) {
  __shared__ double sa[kSlab][kTile];
  __shared__ double sb[kSlab][kTile];
  // tile (bj, bk), bj <= bk, in row-major order of the upper triangle
  int t = blockIdx.x, bj = 0;
  while (t >= nb - bj) {
    t -= nb - bj;
    ++bj;
  }
  const int bk = bj + t;
  const int j0 = bj * kTile, k0 = bk * kTile;
  const bool diag = bj == bk;
  const int tid = threadIdx.x;
  const int tj = tid >> 3, tk = tid & 7;         // outputs (j0 + tj + 8a, k0 + tk + 8b), a, b < 4

  // the column this thread stages: block j for threads 0..31, block k for 32..63
  const int col = tid < kTile ? j0 + tid : k0 + tid - kTile;
  const bool col_ok = col < d;

  double acc[kSub][kSub];
#pragma unroll
  for (int a = 0; a < kSub; ++a)
#pragma unroll
    for (int b = 0; b < kSub; ++b) {
      const int j = j0 + tj + 8 * a, k = k0 + tk + 8 * b;
      acc[a][b] = (j < d && k < d && k >= j) ? gram[(int64_t)j * d + k] : 0.0;
    }
  const bool has_sum = diag && tid < kTile && j0 + tid < d;    // warp 0 of a diagonal tile: one sum column each
  double s_acc = has_sum ? sum[j0 + tid] : 0.0;

  float pre[kSlab];
  auto fetch = [&](int64_t r0) {
#pragma unroll
    for (int r = 0; r < kSlab; ++r) {
      const int64_t i = r0 + r;
      pre[r] = (col_ok && i < n) ? __ldg(z + i * ld + col) : 0.f;
    }
  };
  fetch(0);
  double(*const stage)[kTile] = tid < kTile ? sa : sb;
  const int scol = tid & (kTile - 1);
  for (int64_t r0 = 0; r0 < n; r0 += kSlab) {
#pragma unroll
    for (int r = 0; r < kSlab; ++r) stage[r][scol] = (double)pre[r];
    __syncthreads();
    if (r0 + kSlab < n) fetch(r0 + kSlab);        // in flight while this slab is used
    const int rows = n - r0 < kSlab ? (int)(n - r0) : kSlab;
    if (rows == kSlab) {
#pragma unroll 8
      for (int i = 0; i < kSlab; ++i) {
        double av[kSub], bv[kSub];
#pragma unroll
        for (int a = 0; a < kSub; ++a) av[a] = sa[i][tj + 8 * a];
#pragma unroll
        for (int b = 0; b < kSub; ++b) bv[b] = sb[i][tk + 8 * b];
#pragma unroll
        for (int a = 0; a < kSub; ++a)
#pragma unroll
          for (int b = 0; b < kSub; ++b) acc[a][b] = fma(av[a], bv[b], acc[a][b]);
        if (has_sum) s_acc += sa[i][tid];
      }
    } else {
      for (int i = 0; i < rows; ++i) {              // the last, partial slab: only real rows are added
        double av[kSub], bv[kSub];
#pragma unroll
        for (int a = 0; a < kSub; ++a) av[a] = sa[i][tj + 8 * a];
#pragma unroll
        for (int b = 0; b < kSub; ++b) bv[b] = sb[i][tk + 8 * b];
#pragma unroll
        for (int a = 0; a < kSub; ++a)
#pragma unroll
          for (int b = 0; b < kSub; ++b) acc[a][b] = fma(av[a], bv[b], acc[a][b]);
        if (has_sum) s_acc += sa[i][tid];
      }
    }
    __syncthreads();                                // the slab is rewritten next iteration
  }

#pragma unroll
  for (int a = 0; a < kSub; ++a)
#pragma unroll
    for (int b = 0; b < kSub; ++b) {
      const int j = j0 + tj + 8 * a, k = k0 + tk + 8 * b;
      if (j < d && k < d && k >= j) gram[(int64_t)j * d + k] = acc[a][b];
    }
  if (has_sum) sum[j0 + tid] = s_acc;
}

}  // namespace bvae

using namespace bvae;

extern "C" {

int bvae_latent_moments(const float* z, int64_t n, int32_t d, int64_t ld, double* sum, double* gram, void* stream) {
  BVAE_REQUIRE(n >= 0, BVAE_ERR_SHAPE, "latent_moments: n must be >= 0 (got %lld)", (long long)n);
  BVAE_REQUIRE(d >= 1, BVAE_ERR_SHAPE, "latent_moments: d must be >= 1 (got %d)", (int)d);
  BVAE_REQUIRE(ld >= d, BVAE_ERR_SHAPE, "latent_moments: ld must be >= d (got ld %lld, d %d)", (long long)ld, (int)d);
  BVAE_REQUIRE(((uintptr_t)z & 3) == 0, BVAE_ERR_ALIGN, "latent_moments: z must be 4-byte aligned");
  BVAE_REQUIRE((((uintptr_t)sum | (uintptr_t)gram) & 7) == 0, BVAE_ERR_ALIGN,
               "latent_moments: sum and gram must be 8-byte aligned");
  if (n == 0) return BVAE_OK;
  const int nb = ceil_div(d, kTile);
  const int64_t tiles = (int64_t)nb * (nb + 1) / 2;
  BVAE_REQUIRE(tiles <= 0x7fffffff, BVAE_ERR_SHAPE, "latent_moments: d = %d gives more tiles than one grid holds", (int)d);
  note_kernel("latent_moments_kernel");
  latent_moments_kernel<<<(unsigned)tiles, kMomThreads, 0, (cudaStream_t)stream>>>(z, n, d, ld, nb, sum, gram);
  return check_launch("latent_moments");
}

}  // extern "C"
