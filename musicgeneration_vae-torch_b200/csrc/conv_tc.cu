// conv_tc.cu -- tcgen05 / TMEM / TMA implicit-GEMM kernels for sm_100a.
//
// conv_tc2_kernel (forward + data gradient, operands K-major):
//   D[128 pixels x BN channels] (fp32, TMEM) = sum over (tap, channel block) A[128 x KB] * B[BN x KB]^T
//   A = activation patch: ONE tiled TMA box {KB channels, bw, bh, bn} of an NHWC view per (tap, channel block);
//       the tap shift is a coordinate offset, padding is TMA out-of-bounds zero fill, a strided (stride-2 / k==s)
//       access is a view whose base pointer and strides select the sub-lattice -- no im2col buffer, no gather code.
//   B = packed bf16 weights [Cout][tap][C], one 2-D TMA box {KB, BN}.
//   Both land in shared memory in the canonical 128B (KB=64) / 64B (KB=32) swizzled K-major layout, are consumed by
//   tcgen05.mma.cta_group::1.kind::f16 (M=128, N=BN, K=16) issued by one thread, accumulate in TMEM and are read
//   back with tcgen05.ld for the fused epilogue (bias, (Leaky)ReLU, addend, ReLU-backward mask, bf16/fp32 store
//   with the phase's output stride).
//
// wgrad_tc_kernel (weight gradient, operands MN-major):
//   D_tap[128 anchor channels x NS shifted channels] = sum over pixel blocks  Anchor[pix x 128]^T * Shifted_tap[pix x NS]
//   the contraction index (pixels) is the slow axis of both NHWC tensors, so both operands are MN-major; the same
//   pixel-box TMA loads feed it.  Split over pixel ranges across CTAs, reduced with fp32 red.global.add into the
//   parameter-layout gradient.
#include <cuda.h>
#include <stdlib.h>
#include <mutex>
#include <unordered_map>
#include "common.cuh"

namespace bvae {

// ---------------------------------------------------------------------------------------------------------
// PTX wrappers
// ---------------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  const uint32_t a = smem_u32(bar);
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "WAIT_LOOP:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra DONE;\n\t"
      "bra WAIT_LOOP;\n\t"
      "DONE:\n\t"
      "}" ::"r"(a), "r"(parity) : "memory");
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1) {
  asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
               ::"r"(smem_u32(dst)), "l"((uint64_t)map), "r"(smem_u32(bar)), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void tma_load_4d(void* dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1, int c2,
                                            int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
      ::"r"(smem_u32(dst)), "l"((uint64_t)map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3) : "memory");
}
__device__ __forceinline__ void tma_load_5d(void* dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1, int c2, int c3,
                                            int c4) {
  asm volatile(
      "cp.async.bulk.tensor.5d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6, %7}], [%2];"
      ::"r"(smem_u32(dst)), "l"((uint64_t)map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4) : "memory");
}
// shared -> global tiled store (bulk async group); out-of-bounds elements of the box are clipped
__device__ __forceinline__ void tma_store_4d(const CUtensorMap* map, const void* src, int c0, int c1, int c2, int c3) {
  asm volatile("cp.async.bulk.tensor.4d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5}], [%1];"
               ::"l"((uint64_t)map), "r"(smem_u32(src)), "r"(c0), "r"(c1), "r"(c2), "r"(c3) : "memory");
}
__device__ __forceinline__ void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void tma_store_wait_read() { asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory"); }
__device__ __forceinline__ void tma_store_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void epi_bar_sync(int group = 0) { asm volatile("bar.sync %0, 128;" ::"r"(1 + group) : "memory"); }
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* map) {
  asm volatile("prefetch.tensormap [%0];" ::"l"((uint64_t)map) : "memory");
}

__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

template <int COLS>
__device__ __forceinline__ void tmem_alloc(uint32_t* slot) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(slot)), "n"(COLS) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
template <int COLS>
__device__ __forceinline__ void tmem_dealloc(uint32_t addr) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(addr), "n"(COLS) : "memory");
}
// one lane of a CONVERGED warp (the tcgen05 issue sites sit under this predicate so that ptxas sees a single-lane
// region and does not wrap every MMA in its per-active-lane election loop)
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "elect.sync _|p, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t"
      "}" : "=r"(pred));
  return pred != 0;
}
// D[tmem] (+)= A[smem desc] * B[smem desc]
__device__ __forceinline__ void umma_f16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t acc) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}" ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(acc) : "memory");
}
// NK consecutive K = 16 steps in ONE asm statement: the descriptors advance by STEP (encoded >> 4 units) per step.
// A single statement costs one elect/convergence wrapper in SASS instead of NK -- for N <= 64 tiles the issuing thread's
// own instruction stream, not the tensor pipe, limits the MMA rate.
template <int NK, int STEP>
__device__ __forceinline__ void umma_f16_steps(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t acc) {
  static_assert(NK == 2 || NK == 4, "NK");
  if (NK == 4) {
    asm volatile(
        "{\n\t"
        ".reg .pred p, q;\n\t"
        ".reg .b64 a1, a2, a3, b1, b2, b3;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "setp.eq.b32 q, 0, 0;\n\t"
        "add.u64 a1, %1, %5;\n\t"
        "add.u64 b1, %2, %5;\n\t"
        "add.u64 a2, %1, %6;\n\t"
        "add.u64 b2, %2, %6;\n\t"
        "add.u64 a3, %1, %7;\n\t"
        "add.u64 b3, %2, %7;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], a1, b1, %3, q;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], a2, b2, %3, q;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], a3, b3, %3, q;\n\t"
        "}" ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(acc), "n"(STEP), "n"(2 * STEP), "n"(3 * STEP) : "memory");
  } else {
    asm volatile(
        "{\n\t"
        ".reg .pred p, q;\n\t"
        ".reg .b64 a1, b1;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "setp.eq.b32 q, 0, 0;\n\t"
        "add.u64 a1, %1, %5;\n\t"
        "add.u64 b1, %2, %5;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], a1, b1, %3, q;\n\t"
        "}" ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(acc), "n"(STEP) : "memory");
  }
}
// arrive on an mbarrier once all previously issued tcgen05.mma of this thread have completed
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// 32 lanes x 32 consecutive fp32 columns -> 32 registers per thread
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t* v) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),
        "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),
        "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// shared-memory matrix descriptor (cute::UMMA::SmemDescriptor): start>>4 [0,14) | LBO>>4 [16,30) | SBO>>4 [32,46) |
// version=1 [46,48) | layout type [61,64)  (2 = SWIZZLE_128B, 4 = SWIZZLE_64B)
__device__ __forceinline__ uint64_t make_sdesc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes, uint32_t layout) {
  return (uint64_t)((saddr >> 4) & 0x3FFF) | ((uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16) |
         ((uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32) | (1ull << 46) | ((uint64_t)layout << 61);
}
// instruction descriptor (cute::UMMA::InstrDescriptor) for kind::f16, bf16 x bf16 -> fp32
__host__ __device__ constexpr uint32_t make_idesc(int M, int N, int a_mn_major, int b_mn_major) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)a_mn_major << 15) | ((uint32_t)b_mn_major << 16) |
         ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

// ---------------------------------------------------------------------------------------------------------
// parameters (passed as one __grid_constant__ struct; tensor maps must stay 64-byte aligned)
// ---------------------------------------------------------------------------------------------------------
constexpr int MAX_VIEWS = 6;

struct alignas(64) ConvTcParams {
  CUtensorMap amap[MAX_VIEWS];
  CUtensorMap bmap;
  int tap_view[BVAE_MAX_TAPS];
  int tap_ex[BVAE_MAX_TAPS];
  int tap_ey[BVAE_MAX_TAPS];
  int ntaps, kchunks, C;
  int bw, bh, bn, tiles_w, tiles_h, tiles_n, n_tiles;
  int N, QH, QW, Cout;
  int nphase;                                   // >= 1
  int ph_tap0[BVAE_MAX_PHASES], ph_ntaps[BVAE_MAX_PHASES], ph_ooy[BVAE_MAX_PHASES], ph_oox[BVAE_MAX_PHASES];
  int ph_QH[BVAE_MAX_PHASES], ph_QW[BVAE_MAX_PHASES];
  void* y;
  const float* bias;
  const void* addend;
  const void* mask;
  void* stats;                      // fused InstanceNorm statistics (see bvae_conv_desc.stats) or null
  int OH, OW, y_pitch, osy, osx, ooy, oox, add_pitch, mask_pitch, act, out_f32;
  float slope, mask_slope;
  // halo mode (stride-1 multi-tap layers with resident weights): ONE activation tile with its halo is loaded per
  // (output tile, K chunk) and every tap reads it through a row-shifted shared-memory descriptor
  // TMA-store epilogue (fp32 outputs, BN <= 128): one output tensor map per phase, box {32 floats, bw, bh, bn}
  CUtensorMap ymap[BVAE_MAX_PHASES];
  int tma_store;
  int halo, halo_x0, halo_y0, halo_rows, halo_stage, halo_stages;
  int halo_shift[BVAE_MAX_TAPS];
};

// Column reduction over the 32 rows a warp holds (one row per lane, 32 columns per lane): butterfly in which every
// step halves the number of columns a lane is responsible for; after 5 steps lane l holds the result of column l.
template <typename Op>
__device__ __forceinline__ float warp_col_reduce(float (&v)[32], Op op) {
  const int lane = threadIdx.x & 31;
#pragma unroll
  for (int s = 16; s >= 1; s >>= 1) {
    const bool up = (lane & s) != 0;
#pragma unroll
    for (int i = 0; i < s; ++i) {
      const float mine = up ? v[i + s] : v[i];
      const float other = up ? v[i] : v[i + s];
      v[i] = op(mine, __shfl_xor_sync(0xffffffffu, other, s));
    }
  }
  return v[0];
}

// ---------------------------------------------------------------------------------------------------------
// forward / data-gradient kernel, persistent: one CTA per SM loops over output tiles.  256 threads: warp 0 = TMA
// producer, warp 1 = MMA issuer, warp 2 = TMEM allocator, warps 4..7 = epilogue.  Two TMEM accumulator buffers (2 x BN
// columns) let the epilogue of tile i overlap the main loop of tile i+1; barrier init / TMEM allocation are paid once per
// CTA.
// ---------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}

// BRES: the whole weight operand (all taps x K chunks of the single N tile) is loaded ONCE per CTA and stays resident in
// shared memory; the pipeline then streams activation tiles only (small-channel layers are L2-bandwidth bound and the
// weights were a third of their traffic).
// Narrow tiles (BN <= 64) have main loops of 0.2-0.6 us while one pass of the epilogue (accumulator wait, tcgen05.ld, two
// named barriers, slab write, TMA store) takes about 1.5 us (measured: 23 040 tiles of 32->32 3x3 at 512 bars in 246 us
// = 1.58 us per tile and SM at 3 % tensor-pipe and 30 % DRAM utilisation).  They therefore get TWO epilogue groups of four
// warps (384 threads): group g drains accumulator buffer g, i.e. the CTA's even / odd tiles, through its own pair of output
// slabs and its own named barrier, so two epilogues run concurrently next to the main loop of a third tile.
template <int BN>
struct ConvTc2Cfg {
  static constexpr int EG = BN <= 64 ? 2 : 1;            // epilogue groups
  static constexpr int THREADS = 128 + 128 * EG;
};

template <int KB, int BN, int STAGES, bool BRES>
__global__ void __launch_bounds__(ConvTc2Cfg<BN>::THREADS, 1) conv_tc2_kernel(const __grid_constant__ ConvTcParams p) {
  constexpr int EG = ConvTc2Cfg<BN>::EG;
  constexpr int A_BYTES = 128 * KB * 2;
  constexpr int B_BYTES = BN * KB * 2;
  constexpr int STAGE_BYTES = BRES ? A_BYTES : A_BYTES + B_BYTES;
  constexpr int ACC_COLS = BN <= 32 ? 32 : (BN <= 64 ? 64 : (BN <= 128 ? 128 : 256));
  constexpr int TMEM_COLS = 2 * ACC_COLS;
  constexpr uint32_t LAYOUT = KB == 64 ? 2u : 4u;
  constexpr uint32_t SBO = 8 * KB * 2;
  constexpr uint32_t IDESC = make_idesc(128, BN, 0, 0);

  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem_al = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  uint8_t* bres = smem_al;                                       // [ntaps * kchunks][BN x KB] resident weights (BRES)
  uint8_t* smem = smem_al + (BRES ? p.ntaps * p.kchunks * B_BYTES : 0);
  uint64_t* full_bar = (uint64_t*)(smem + STAGES * STAGE_BYTES);
  uint64_t* empty_bar = full_bar + STAGES;
  uint64_t* tfull = empty_bar + STAGES;       // [2]
  uint64_t* tempty = tfull + 2;               // [2]
  uint64_t* bres_bar = tempty + 2;
  uint32_t* tmem_slot = (uint32_t*)(bres_bar + 1);
  // two 16 KB slabs [128 rows][32 floats], 128B-swizzled, for the TMA-store epilogue
  uint8_t* ystage = (uint8_t*)(((uintptr_t)(tmem_slot + 4) + 1023) & ~(uintptr_t)1023);
  const bool halo = BRES && KB == 64 && p.halo;
  const uint32_t nst = halo ? (uint32_t)p.halo_stages : (uint32_t)STAGES;      // ring depth / stage size in use
  const uint32_t stage_bytes = halo ? (uint32_t)p.halo_stage : (uint32_t)STAGE_BYTES;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int m_tiles = p.tiles_w * p.tiles_h * p.tiles_n;
  const int total = m_tiles * p.nphase * p.n_tiles;     // tile order: N tile fastest, then phase, then the pixel box

  if (warp == 0 && lane == 0) {
    for (int s = 0; s < STAGES; ++s) { mbar_init(full_bar + s, 1); mbar_init(empty_bar + s, 1); }
    for (int b = 0; b < 2; ++b) { mbar_init(tfull + b, 1); mbar_init(tempty + b, 128); }
    mbar_init(bres_bar, 1);
    fence_barrier_init();
    tma_prefetch_desc(&p.bmap);
    tma_prefetch_desc(&p.amap[0]);
  }
  if (warp == 2) tmem_alloc<TMEM_COLS>(tmem_slot);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0 && lane == 0) {
    // ---------------- TMA producer ----------------
    const uint32_t tx = halo ? (uint32_t)(p.halo_rows * KB * 2) : (uint32_t)(p.bn * p.bh * p.bw * KB * 2 + (BRES ? 0 : B_BYTES));
    if (BRES) {
      mbar_expect_tx(bres_bar, (uint32_t)(p.ntaps * p.kchunks * B_BYTES));
      for (int t = 0; t < p.ntaps; ++t)
        for (int kc = 0; kc < p.kchunks; ++kc)
          tma_load_2d(bres + (t * p.kchunks + kc) * B_BYTES, &p.bmap, bres_bar, t * p.C + kc * KB, 0);
    }
    uint32_t s = 0, par = 0;
    for (int tile = blockIdx.x; tile < total; tile += gridDim.x) {
      const int n_tile = tile % p.n_tiles;
      int m_tile = tile / p.n_tiles;
      int ph = m_tile % p.nphase; m_tile /= p.nphase;
      ph = (ph + m_tile) % p.nphase;      // rotate: a static round-robin must not pin a CTA to one phase (unequal tap counts)
      const int tw = m_tile % p.tiles_w; m_tile /= p.tiles_w;
      const int th = m_tile % p.tiles_h;
      const int tn = m_tile / p.tiles_h;
      if (halo) {
        for (int kc = 0; kc < p.kchunks; ++kc) {
          mbar_wait(empty_bar + s, par ^ 1u);
          mbar_expect_tx(full_bar + s, tx);
          tma_load_4d(smem + s * stage_bytes, &p.amap[0], full_bar + s, kc * KB, p.halo_x0, th * p.bh + p.halo_y0, tn);
          if (++s == nst) { s = 0; par ^= 1u; }
        }
        continue;
      }
      for (int t = p.ph_tap0[ph]; t < p.ph_tap0[ph] + p.ph_ntaps[ph]; ++t) {
        const CUtensorMap* am = &p.amap[p.tap_view[t]];
        const int cw = tw * p.bw + p.tap_ex[t], ch = th * p.bh + p.tap_ey[t], cn = tn * p.bn;
        for (int kc = 0; kc < p.kchunks; ++kc) {
          mbar_wait(empty_bar + s, par ^ 1u);
          mbar_expect_tx(full_bar + s, tx);
          uint8_t* sa = smem + s * stage_bytes;
          tma_load_4d(sa, am, full_bar + s, kc * KB, cw, ch, cn);
          if (!BRES) tma_load_2d(sa + A_BYTES, &p.bmap, full_bar + s, t * p.C + kc * KB, n_tile * BN);
          if (++s == nst) { s = 0; par ^= 1u; }
        }
      }
    }
  } else if (warp == 1) {
    // ---------------- MMA issuer: the whole warp walks the loop, one elected lane issues ----------------
    uint32_t s = 0, par = 0, ti = 0;
    if (BRES) { mbar_wait(bres_bar, 0); tc_fence_after(); }
    for (int tile = blockIdx.x; tile < total; tile += gridDim.x, ++ti) {
      const uint32_t ab = ti & 1u, aph = (ti >> 1) & 1u;
      mbar_wait(tempty + ab, aph ^ 1u);            // epilogue has drained this accumulator buffer
      tc_fence_after();
      const uint32_t tacc = tmem_base + ab * ACC_COLS;
      const int rest = tile / p.n_tiles;
      const int phase = (rest % p.nphase + rest / p.nphase) % p.nphase;
      const int KT = p.ph_ntaps[phase] * p.kchunks;
      const uint32_t bres0 = smem_u32(bres) + (uint32_t)(p.ph_tap0[phase] * p.kchunks) * B_BYTES;
      if (halo) {
        for (int kc = 0; kc < p.kchunks; ++kc) {
          mbar_wait(full_bar + s, par);
          tc_fence_after();
          const uint32_t sa = smem_u32(smem + s * stage_bytes);
          if (elect_one()) {
            for (int t = 0; t < p.ntaps; ++t) {
              // tap t = the same tile, p.halo_shift[t] pixel rows (128 B each) further on.  Measured on B200: the 128B
              // swizzle XOR is taken from the absolute shared-memory address bits [7,10) - exactly how TMA wrote the
              // tile - so a start address that is not 1024-byte aligned needs NO descriptor base offset (setting
              // (addr >> 7) & 7 there gives wrong results).
              const uint64_t adesc = make_sdesc(sa + (uint32_t)p.halo_shift[t] * 128u, 16, SBO, LAYOUT);
              const uint64_t bdesc = make_sdesc(bres0 + (uint32_t)(t * p.kchunks + kc) * B_BYTES, 16, SBO, LAYOUT);
              umma_f16_steps<KB / 16, 2>(tacc, adesc, bdesc, IDESC, (kc | t) ? 1u : 0u);
            }
            umma_commit(empty_bar + s);
          }
          __syncwarp();
          if (++s == nst) { s = 0; par ^= 1u; }
        }
        if (elect_one()) umma_commit(tfull + ab);
        __syncwarp();
        continue;
      }
      for (int kb = 0; kb < KT; ++kb) {
        mbar_wait(full_bar + s, par);
        tc_fence_after();
        const uint32_t sa = smem_u32(smem + s * stage_bytes);
        if (elect_one()) {
          const uint64_t adesc = make_sdesc(sa, 16, SBO, LAYOUT);
          const uint64_t bdesc = make_sdesc(BRES ? bres0 + (uint32_t)kb * B_BYTES : sa + A_BYTES, 16, SBO, LAYOUT);
          umma_f16_steps<KB / 16, 2>(tacc, adesc, bdesc, IDESC, kb ? 1u : 0u);
          umma_commit(empty_bar + s);
        }
        __syncwarp();
        if (++s == nst) { s = 0; par ^= 1u; }
      }
      if (elect_one()) umma_commit(tfull + ab);
      __syncwarp();
    }
  } else if (warp >= 4) {
    // ---------------- epilogue warps: TMEM -> registers -> global ----------------
    const int wq = warp & 3;                       // TMEM lane quarter this warp may access (= warp id % 4)
    const uint32_t eg = (uint32_t)(warp - 4) >> 2; // epilogue group: drains accumulator buffer eg (EG == 2) or both
    uint8_t* const yslabs = ystage + eg * 32768u;  // this group's two output slabs
    uint32_t gsl = 0;                              // slabs this group has handed to TMA so far
    const int r = wq * 32 + lane;
    const int rows_box = p.bn * p.bh * p.bw;
    const int nn = r / (p.bh * p.bw), hh = (r / p.bw) % p.bh, ww = r % p.bw;
    uint32_t ti = 0;
    for (int tile = blockIdx.x; tile < total; tile += gridDim.x, ++ti) {
      const uint32_t ab = ti & 1u, aph = (ti >> 1) & 1u;
      if (EG == 2 && ab != eg) continue;  // the other group's tile
      const int n_tile = tile % p.n_tiles;
      int m_tile = tile / p.n_tiles;
      int ph = m_tile % p.nphase; m_tile /= p.nphase;
      ph = (ph + m_tile) % p.nphase;      // rotate: a static round-robin must not pin a CTA to one phase (unequal tap counts)
      const int tw = m_tile % p.tiles_w; m_tile /= p.tiles_w;
      const int th = m_tile % p.tiles_h;
      const int tn = m_tile / p.tiles_h;
      const int n = tn * p.bn + nn, qy = th * p.bh + hh, qx = tw * p.bw + ww;
      const bool valid = r < rows_box && n < p.N && qy < p.ph_QH[ph] && qx < p.ph_QW[ph];
      const int64_t opix = ((int64_t)n * p.OH + (qy * p.osy + p.ph_ooy[ph])) * p.OW + (qx * p.osx + p.ph_oox[ph]);
      const int col0 = n_tile * BN;
      // narrow tiles (BN <= 64) have short main loops: fetch the activation mask / bf16 addend of this row BEFORE
      // waiting for the accumulator so that their latency overlaps the MMAs instead of serialising the epilogue
      constexpr bool PRE = BN <= 64;
      constexpr int NPRE = PRE ? BN / 8 : 1;
      bf16x8 pre_m[NPRE], pre_a[NPRE];
      const bool pre_mask = PRE && p.mask && valid && !p.stats;
      const bool pre_add = PRE && p.addend && !p.out_f32 && valid && !p.stats;
      if (pre_mask) {
        const bf16* mp = (const bf16*)p.mask + opix * p.mask_pitch + col0;
#pragma unroll
        for (int i = 0; i < NPRE; ++i) pre_m[i] = ldg8(mp + 8 * i);
      }
      if (pre_add) {
        const bf16* ap = (const bf16*)p.addend + opix * p.add_pitch + col0;
#pragma unroll
        for (int i = 0; i < NPRE; ++i) pre_a[i] = ldg8(ap + 8 * i);
      }
      mbar_wait(tfull + ab, aph);
      tc_fence_after();
      const uint32_t tacc = tmem_base + ab * ACC_COLS + ((uint32_t)(wq * 32) << 16);
      if (BN <= 128 && p.tma_store) {
        // fp32 output through shared memory and one tiled TMA store per 128-byte-wide slab (32 columns): the direct
        // path issues, per warp instruction, 32 separate 16-byte requests to 32 different rows (2048 L1 requests per
        // 128x64 fp32 tile), which made the epilogue the longest stage of the small-K layers.  Rows and columns outside
        // the output are clipped by the store.
#pragma unroll(PRE ? 2 : 1)
        for (int c0 = 0; c0 < BN; c0 += 32) {
          uint32_t v[32];
          tmem_ld32(tacc + (uint32_t)c0, v);
          if (c0 + 32 >= BN) { tc_fence_before(); mbar_arrive(tempty + ab); }     // accumulator drained
          uint8_t* slab = yslabs + (gsl & 1u) * 16384u;
          float f[32];
#pragma unroll
          for (int i = 0; i < 32; ++i) f[i] = __uint_as_float(v[i]);
          if (p.bias) {
#pragma unroll
            for (int i = 0; i < 32; i += 4) {
              const float4 b4 = __ldg(reinterpret_cast<const float4*>(p.bias + col0 + c0 + i));
              f[i] += b4.x; f[i + 1] += b4.y; f[i + 2] += b4.z; f[i + 3] += b4.w;
            }
          }
          if (p.act) {
#pragma unroll
            for (int i = 0; i < 32; ++i) f[i] = act_fwd(f[i], p.slope);
          }
          if (p.addend && valid) {
            const float* ap = (const float*)p.addend + opix * p.add_pitch + col0 + c0;
#pragma unroll
            for (int i = 0; i < 32; i += 4) {
              const float4 a = *reinterpret_cast<const float4*>(ap + i);
              f[i] += a.x; f[i + 1] += a.y; f[i + 2] += a.z; f[i + 3] += a.w;
            }
          }
          if (p.mask && valid) {
            const bf16* mp = (const bf16*)p.mask + opix * p.mask_pitch + col0 + c0;
#pragma unroll
            for (int i = 0; i < 32; i += 8) {
              float a[8];
              unpack8((PRE && pre_mask) ? pre_m[PRE ? ((c0 + i) / 8) % NPRE : 0] : ldg8(mp + i), a);
#pragma unroll
              for (int k = 0; k < 8; ++k) f[i + k] *= (a[k] > 0.f) ? 1.f : p.mask_slope;
            }
          }
          uint8_t* row = slab + r * 128;
          const int sw = r & 7;
          // the store issued from this slab buffer two slabs ago must have finished reading it
          if (r == 0) tma_store_wait_read<1>();
          epi_bar_sync(eg);
#pragma unroll
          for (int j = 0; j < 8; ++j)
            *reinterpret_cast<float4*>(row + ((j ^ sw) << 4)) = make_float4(f[4 * j], f[4 * j + 1], f[4 * j + 2], f[4 * j + 3]);
          fence_proxy_async();
          epi_bar_sync(eg);
          if (r == 0) {
            tma_store_4d(&p.ymap[ph], slab, col0 + c0, tw * p.bw, th * p.bh, tn * p.bn);
            tma_store_commit();
          }
          ++gsl;
        }
        continue;
      }
#pragma unroll(PRE ? 2 : 1)
      for (int c0 = 0; c0 < BN; c0 += 32) {
        uint32_t v[32];
        tmem_ld32(tacc + (uint32_t)c0, v);
        if (p.stats) {
          // raw fp32 output in front of an InstanceNorm: store it and reduce this warp's 32 rows per column
          // (sum, sum of squares, max, min) -> one double / key atomic per column; the tile lies inside sample tn
          float f[32], g[32];
#pragma unroll
          for (int i = 0; i < 32; ++i) f[i] = __uint_as_float(v[i]);
          if (p.bias) {
#pragma unroll
            for (int i = 0; i < 32; i += 4) {
              const float4 b4 = __ldg(reinterpret_cast<const float4*>(p.bias + col0 + c0 + i));
              f[i] += b4.x; f[i + 1] += b4.y; f[i + 2] += b4.z; f[i + 3] += b4.w;
            }
          }
          if (valid) {
            float* yp = (float*)p.y + opix * p.y_pitch + col0 + c0;
#pragma unroll
            for (int i = 0; i < 32; i += 4) *reinterpret_cast<float4*>(yp + i) = make_float4(f[i], f[i + 1], f[i + 2], f[i + 3]);
          }
#pragma unroll
          for (int i = 0; i < 32; ++i) g[i] = valid ? f[i] : 0.f;
          const float s1 = warp_col_reduce(g, [](float a, float b) { return a + b; });
#pragma unroll
          for (int i = 0; i < 32; ++i) g[i] = valid ? f[i] * f[i] : 0.f;
          const float s2 = warp_col_reduce(g, [](float a, float b) { return a + b; });
#pragma unroll
          for (int i = 0; i < 32; ++i) g[i] = valid ? f[i] : -INFINITY;
          const float mx = warp_col_reduce(g, [](float a, float b) { return fmaxf(a, b); });
#pragma unroll
          for (int i = 0; i < 32; ++i) g[i] = valid ? -f[i] : -INFINITY;
          const float mn = warp_col_reduce(g, [](float a, float b) { return fmaxf(a, b); });     // max of -x
          const long long NC = (long long)p.N * p.Cout;
          const long long o = (long long)tn * p.Cout + col0 + c0 + lane;
          double* sd = (double*)p.stats;
          atomicAdd(sd + o, (double)s1);
          atomicAdd(sd + NC + o, (double)s2);
          uint32_t* kk = (uint32_t*)(sd + 2 * NC);
          atomicMax(kk + o, f2ord(mx));
          atomicMax(kk + NC + o, f2ord(mn));
          continue;
        }
        if (!valid) continue;
        float f[32];
#pragma unroll
        for (int i = 0; i < 32; ++i) f[i] = __uint_as_float(v[i]);
        if (p.bias) {
#pragma unroll
          for (int i = 0; i < 32; i += 4) {
            const float4 b4 = __ldg(reinterpret_cast<const float4*>(p.bias + col0 + c0 + i));
            f[i] += b4.x; f[i + 1] += b4.y; f[i + 2] += b4.z; f[i + 3] += b4.w;
          }
        }
        if (p.act) {
#pragma unroll
          for (int i = 0; i < 32; ++i) f[i] = act_fwd(f[i], p.slope);
        }
        if (p.addend) {
          if (p.out_f32) {
            const float* ap = (const float*)p.addend + opix * p.add_pitch + col0 + c0;
#pragma unroll
            for (int i = 0; i < 32; i += 4) {
              const float4 a = *reinterpret_cast<const float4*>(ap + i);
              f[i] += a.x; f[i + 1] += a.y; f[i + 2] += a.z; f[i + 3] += a.w;
            }
          } else {
            const bf16* ap = (const bf16*)p.addend + opix * p.add_pitch + col0 + c0;
#pragma unroll
            for (int i = 0; i < 32; i += 8) {
              float a[8];
              unpack8(PRE ? pre_a[PRE ? (c0 + i) / 8 : 0] : ldg8(ap + i), a);
#pragma unroll
              for (int k = 0; k < 8; ++k) f[i + k] += a[k];
            }
          }
        }
        if (p.mask) {
          const bf16* mp = (const bf16*)p.mask + opix * p.mask_pitch + col0 + c0;
#pragma unroll
          for (int i = 0; i < 32; i += 8) {
            float a[8];
            unpack8(PRE ? pre_m[PRE ? (c0 + i) / 8 : 0] : ldg8(mp + i), a);
#pragma unroll
            for (int k = 0; k < 8; ++k) f[i + k] *= (a[k] > 0.f) ? 1.f : p.mask_slope;
          }
        }
        if (p.out_f32) {
          float* yp = (float*)p.y + opix * p.y_pitch + col0 + c0;
#pragma unroll
          for (int i = 0; i < 32; i += 4) *reinterpret_cast<float4*>(yp + i) = make_float4(f[i], f[i + 1], f[i + 2], f[i + 3]);
        } else {
          bf16* yp = (bf16*)p.y + opix * p.y_pitch + col0 + c0;
#pragma unroll
          for (int i = 0; i < 32; i += 8) stg8(yp + i, pack8(f + i));
        }
      }
      tc_fence_before();
      mbar_arrive(tempty + ab);                    // 128 arrivals release the accumulator buffer
    }
  }
  if ((threadIdx.x == 128 || (EG == 2 && threadIdx.x == 256)) && BN <= 128 && p.tma_store) tma_store_wait_all();   // r == 0 of each epilogue group
  tc_fence_before();
  __syncthreads();
  if (warp == 2) tmem_dealloc<TMEM_COLS>(tmem_base);
}

// ---------------------------------------------------------------------------------------------------------
// weight-gradient kernel
// ---------------------------------------------------------------------------------------------------------
struct alignas(64) WgradTcParams {
  CUtensorMap amap;                 // anchor tensor, box {64 ch, bw, bh, bn}
  CUtensorMap smap[MAX_VIEWS];      // shifted tensor views, same box
  int tap_view[BVAE_MAX_TAPS];
  int tap_ex[BVAE_MAX_TAPS];
  int tap_ey[BVAE_MAX_TAPS];
  int tap_idx[BVAE_MAX_TAPS];
  int ntaps, T, tpc, tap_groups;    // taps per CTA, number of tap groups
  int bw, bh, bn, chunks_w, chunks_h, chunks_n, nchunks, chunks_per_split, splits;
  int a_atoms;                      // 64-channel atoms of the anchor tile actually loaded (1 or 2)
  int ra_tiles, rs_tiles;
  int wt;                           // 1: "wide TMA" -- amap / smap are 5-D {64 ch, W, H, N, channel block} maps, one request per operand
  int wt_stages, wt_stage_bytes;    // WT: ring depth (2..4) and bytes per stage = atoms * rows_box * 128 (packed atoms)
  int Ca, Cs;
  float* dw;                        // destination of the reduction (parameter gradient or packed scratch)
  long long s_ra, s_t;              // element strides of the anchor channel / the tap; the shifted channel stride is
  int s_rs;                         // 1 (vector reductions) or T (scalar reductions straight into [ra][rs][tap])
  // halo variant (wgrad_halo_kernel): one shifted-tensor tile with its halo per chunk, taps = row-shifted descriptors
  int h_PW, h_RH, h_rows_a, h_rows_s, h_stage, h_stages, h_x0, h_y0, h_tiles_h;
  int h_shift[BVAE_MAX_TAPS];
};

// CB = channels per swizzle atom (64 -> SWIZZLE_128B, 32 -> SWIZZLE_64B); NS = shifted-channel tile (multiple of
// CB, <= 256); KP = 64 pixel rows per stage
// WT ("wide TMA", 64-channel atoms, boxes of a multiple of 16 pixel rows): ncu on 512->512 3x3 at 6x4 x 512 bars showed the
// MMA warp waiting for data 45 % of the K loop at 33 % L2 and 5 % DRAM utilisation -- ten TMA requests of 6-8 KB per 64-pixel
// stage (2 anchor atoms + 2 taps x 4 shifted atoms) against two requests per stage in conv_tc2, i.e. the request rate, not the
// bytes, is what the two-stage ring cannot hide.  With the channel axis split as a FIFTH tensor-map dimension {64 ch, W, H, N,
// C/64} a box {64, bw, bh, bn, atoms} lands as `atoms` consecutive [rows][64 ch] swizzled tiles: ONE request per operand and
// tap (3 per stage instead of 10).  The tiles are packed (rows_box * 128 B apart, the descriptors' leading-dimension offset),
// every row of every tile is rewritten by each request (out-of-bounds pixels arrive as zeros), so the ring needs no zeroing.
template <int CB, int NS, int STAGES, bool WT = false>
__global__ void __launch_bounds__(128) wgrad_tc_kernel(const __grid_constant__ WgradTcParams p) {
  constexpr int KP = 64;
  constexpr int ROW_BYTES = CB * 2;
  constexpr int ATOM_BYTES = KP * ROW_BYTES;           // [64 pixel rows][CB channels] bf16, swizzled
  constexpr int A_ATOMS = 128 / CB;                    // the MMA always spans M = 128 anchor channels
  constexpr int S_ATOMS = NS / CB;
  constexpr int MAX_TPC = (512 / NS) > BVAE_MAX_TAPS ? BVAE_MAX_TAPS : (512 / NS);
  constexpr int STAGE_BYTES = (A_ATOMS + MAX_TPC * S_ATOMS) * ATOM_BYTES;
  constexpr uint32_t LAYOUT = CB == 64 ? 2u : 4u;
  constexpr uint32_t SBO = 8 * ROW_BYTES;              // 8 pixel rows
  constexpr uint32_t KSTEP = (16 * ROW_BYTES) >> 4;    // 16 pixel rows per MMA, in encoded (>>4) address units

  // WT: the packed atoms make a stage atoms * rows_box * 128 bytes, so boxes of 48 / 32 pixel rows (the 6x4, 3x2, 12x2 maps of
  // the 512 / 1024-channel layers) fit a THIRD / FOURTH ring stage into the same shared memory: the ring depth is a launch
  // parameter there and the barriers sit in front of the ring.
  constexpr int MAXST = WT ? 4 : STAGES;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  const int nst = WT ? p.wt_stages : STAGES;
  const uint32_t stage_bytes = WT ? (uint32_t)p.wt_stage_bytes : (uint32_t)STAGE_BYTES;
  uint8_t* ring = WT ? smem + 1024 : smem;
  uint64_t* full_bar = WT ? (uint64_t*)smem : (uint64_t*)(smem + STAGES * STAGE_BYTES);
  uint64_t* empty_bar = full_bar + MAXST;
  uint64_t* tmem_full = empty_bar + MAXST;
  uint32_t* tmem_slot = (uint32_t*)(tmem_full + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  int b = blockIdx.x;
  const int split = b % p.splits; b /= p.splits;
  const int tg = b % p.tap_groups; b /= p.tap_groups;
  const int rs_tile = b % p.rs_tiles;
  const int ra_tile = b / p.rs_tiles;
  const int tap0 = tg * p.tpc;
  const int ntap = min(p.tpc, p.ntaps - tap0);
  const int ck0 = split * p.chunks_per_split;
  const int ck1 = min(p.nchunks, ck0 + p.chunks_per_split);
  const int rows_box = p.bn * p.bh * p.bw;             // <= 64, the rest of each atom stays zero

  // zero the whole pipeline buffer once: rows a box never writes must contribute exactly 0 to the contraction
  if (!WT) {
    for (int i = threadIdx.x; i < STAGES * STAGE_BYTES / 16; i += 128) reinterpret_cast<uint4*>(smem)[i] = make_uint4(0, 0, 0, 0);
    fence_proxy_async();
  }
  const uint32_t atom_stride = WT ? (uint32_t)(rows_box * ROW_BYTES) : (uint32_t)ATOM_BYTES;   // distance between channel atoms
  if (warp == 0 && lane == 0) {
    for (int s = 0; s < MAXST; ++s) { mbar_init(full_bar + s, 1); mbar_init(empty_bar + s, 1); }
    mbar_init(tmem_full, 1);
    fence_barrier_init();
    tma_prefetch_desc(&p.amap);
  }
  if (warp == 2) tmem_alloc<512>(tmem_slot);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0 && lane == 0) {
    const uint32_t tx = (uint32_t)(rows_box * ROW_BYTES * (p.a_atoms + ntap * S_ATOMS));
    int s = 0;
    uint32_t ph = 0;
    for (int ck = ck0; ck < ck1; ++ck) {
      int q = ck;
      const int cw = (q % p.chunks_w) * p.bw; q /= p.chunks_w;
      const int ch = (q % p.chunks_h) * p.bh;
      const int cn = (q / p.chunks_h) * p.bn;
      mbar_wait(empty_bar + s, ph ^ 1u);
      mbar_expect_tx(full_bar + s, tx);
      uint8_t* st = ring + (uint32_t)s * stage_bytes;
      if (WT) {
        tma_load_5d(st, &p.amap, full_bar + s, 0, cw, ch, cn, ra_tile * A_ATOMS);
        for (int t = 0; t < ntap; ++t) {
          const int tap = tap0 + t;
          tma_load_5d(st + (A_ATOMS + t * S_ATOMS) * atom_stride, &p.smap[p.tap_view[tap]], full_bar + s, 0,
                      cw + p.tap_ex[tap], ch + p.tap_ey[tap], cn, rs_tile * S_ATOMS);
        }
      }
      for (int a = 0; !WT && a < p.a_atoms; ++a)
        tma_load_4d(st + a * ATOM_BYTES, &p.amap, full_bar + s, (ra_tile * A_ATOMS + a) * CB, cw, ch, cn);
      for (int t = 0; !WT && t < ntap; ++t) {
        const int tap = tap0 + t;
        const CUtensorMap* sm = &p.smap[p.tap_view[tap]];
        for (int a = 0; a < S_ATOMS; ++a)
          tma_load_4d(st + (A_ATOMS + t * S_ATOMS + a) * ATOM_BYTES, sm, full_bar + s, rs_tile * NS + a * CB,
                      cw + p.tap_ex[tap], ch + p.tap_ey[tap], cn);
      }
      if (++s == nst) { s = 0; ph ^= 1u; }
    }
  } else if (warp == 1) {
    // the whole warp walks the loop, one elected lane issues (see elect_one)
    const int ksteps = (rows_box + 15) / 16;
    int it = 0, s = 0;
    uint32_t ph = 0;
    for (int ck = ck0; ck < ck1; ++ck, ++it) {
      mbar_wait(full_bar + s, ph);
      tc_fence_after();
      const uint32_t st = smem_u32(ring + (uint32_t)s * stage_bytes);
      if (elect_one()) {
        // MN-major: LBO = distance between CB-channel atoms, SBO = 8 pixel rows
        const uint64_t adesc = make_sdesc(st, atom_stride, SBO, LAYOUT);
        // the atoms of consecutive taps are contiguous in smem and their accumulators are contiguous TMEM columns, so
        // up to 256/NS taps go into ONE instruction with N = taps*NS (A is read once for all of them)
        constexpr int TG = 256 / NS;
        for (int t = 0; t < ntap; t += TG) {
          const int tg = min(TG, ntap - t);
          const uint32_t idesc = make_idesc(128, tg * NS, 1, 1);
          const uint64_t bdesc = make_sdesc(st + (A_ATOMS + t * S_ATOMS) * atom_stride, atom_stride, SBO, LAYOUT);
          if (ksteps == 4) {
            umma_f16_steps<4, (int)KSTEP>(tmem_base + (uint32_t)(t * NS), adesc, bdesc, idesc, it ? 1u : 0u);
          } else {
            for (int j = 0; j < ksteps; ++j)
              umma_f16(tmem_base + (uint32_t)(t * NS), adesc + KSTEP * j, bdesc + KSTEP * j, idesc, (it | j) ? 1u : 0u);
          }
        }
        umma_commit(empty_bar + s);
      }
      __syncwarp();
      if (++s == nst) { s = 0; ph ^= 1u; }
    }
    if (elect_one()) umma_commit(tmem_full);
    __syncwarp();
  }
  __syncwarp();
  mbar_wait(tmem_full, 0);
  tc_fence_after();

  // epilogue: lane = anchor channel, columns = shifted channels; scatter-add into the parameter layout
  const int ra = ra_tile * 128 + threadIdx.x;
  const bool valid = threadIdx.x < p.a_atoms * CB && ra < p.Ca;
  for (int t = 0; t < ntap; ++t) {
    const int tix = p.tap_idx[tap0 + t];
#pragma unroll 1
    for (int c0 = 0; c0 < NS; c0 += 32) {
      uint32_t v[32];
      tmem_ld32(tmem_base + ((uint32_t)(warp * 32) << 16) + (uint32_t)(t * NS + c0), v);
      if (!valid || ck1 <= ck0) continue;
      if (p.s_rs == 1) {
        float* dst = p.dw + (int64_t)ra * p.s_ra + (int64_t)tix * p.s_t + rs_tile * NS + c0;
#pragma unroll
        for (int i = 0; i < 32; i += 4)
          atomicAdd(reinterpret_cast<float4*>(dst + i), make_float4(__uint_as_float(v[i]), __uint_as_float(v[i + 1]),
                                                                   __uint_as_float(v[i + 2]), __uint_as_float(v[i + 3])));
      } else {
        float* dst = p.dw + ((int64_t)ra * p.Cs + rs_tile * NS + c0) * p.T + tix;
#pragma unroll
        for (int i = 0; i < 32; ++i) atomicAdd(dst + (int64_t)i * p.T, __uint_as_float(v[i]));
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 2) tmem_dealloc<512>(tmem_base);
}

// Halo variant for 64 -> 64 channel stride-1 layers.  The generic kernel wastes half of every MMA there (M = 128 rows
// for 64 anchor channels) and re-loads the shifted tensor once per tap; this one
//   * flattens a chunk to RH image rows of the PADDED width PW = AW + (dx_max - dx_min): the anchor tile is loaded
//     with its padding columns out of bounds (= zero, so they contribute nothing) and the shifted tensor is loaded ONCE
//     per chunk as (RH + dy_max - dy_min) padded rows; tap (dy, dx) is that tile (dy - dy_min) * PW + (dx - dx_min)
//     pixel rows further on, i.e. a start-address shift of the MN-major descriptor (the 128B swizzle is a function of
//     the absolute shared-memory address, see conv_tc2_kernel);
//   * makes the SHIFTED tensor the M operand and stacks TWO taps in it: the two 64-channel blocks of the M = 128
//     operand are the same tile at two row shifts, expressed through the descriptor's leading-dimension byte offset.
//     D[(tap of the pair, shifted channel)][anchor channel] fills all 128 lanes, N = 64 anchor channels.
__global__ void __launch_bounds__(128) wgrad_halo_kernel(const __grid_constant__ WgradTcParams p) {
  constexpr int ROW = 128;                              // bytes per pixel row (64 bf16 channels)
  constexpr int ATOM_BYTES = 64 * ROW;                  // anchor: [64 pixel rows][64 channels]
  constexpr uint32_t SBO = 8 * ROW;
  constexpr uint32_t KSTEP = (16 * ROW) >> 4;
  constexpr uint32_t IDESC = make_idesc(128, 64, 1, 1);
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  const int STAGES = p.h_stages, STAGE_BYTES = p.h_stage;
  uint64_t* full_bar = (uint64_t*)(smem + STAGES * STAGE_BYTES);
  uint64_t* empty_bar = full_bar + STAGES;
  uint64_t* tmem_full = empty_bar + STAGES;
  uint32_t* tmem_slot = (uint32_t*)(tmem_full + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int split = blockIdx.x;
  const int npairs = (p.ntaps + 1) >> 1;
  const int ck0 = split * p.chunks_per_split;
  const int ck1 = min(p.nchunks, ck0 + p.chunks_per_split);

  // zero the pipeline buffer once: anchor rows a box never writes must be 0, and whatever a shifted descriptor reads
  // past the loaded tile must at least be finite
  for (int i = threadIdx.x; i < STAGES * STAGE_BYTES / 16; i += 128) reinterpret_cast<uint4*>(smem)[i] = make_uint4(0, 0, 0, 0);
  fence_proxy_async();
  if (warp == 0 && lane == 0) {
    for (int s = 0; s < STAGES; ++s) { mbar_init(full_bar + s, 1); mbar_init(empty_bar + s, 1); }
    mbar_init(tmem_full, 1);
    fence_barrier_init();
    tma_prefetch_desc(&p.amap);
    tma_prefetch_desc(&p.smap[0]);
  }
  if (warp == 2) tmem_alloc<512>(tmem_slot);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0 && lane == 0) {
    const uint32_t tx = (uint32_t)((p.h_rows_a + p.h_rows_s) * ROW);
    int s = 0; uint32_t par = 0;
    for (int ck = ck0; ck < ck1; ++ck) {
      const int th = ck % p.h_tiles_h, n = ck / p.h_tiles_h;
      mbar_wait(empty_bar + s, par ^ 1u);
      mbar_expect_tx(full_bar + s, tx);
      uint8_t* st = smem + s * STAGE_BYTES;
      tma_load_4d(st, &p.amap, full_bar + s, 0, 0, th * p.h_RH, n);
      tma_load_4d(st + ATOM_BYTES, &p.smap[0], full_bar + s, 0, p.h_x0, th * p.h_RH + p.h_y0, n);
      if (++s == STAGES) { s = 0; par ^= 1u; }
    }
  } else if (warp == 1) {
    const int ksteps = (p.h_rows_a + 15) / 16;
    int s = 0; uint32_t par = 0;
    for (int ck = ck0; ck < ck1; ++ck) {
      mbar_wait(full_bar + s, par);
      tc_fence_after();
      const uint32_t st = smem_u32(smem + s * STAGE_BYTES);
      if (elect_one()) {
        const uint64_t bdesc = make_sdesc(st, ATOM_BYTES, SBO, 2u);               // anchor: N = 64 channels, one block
        for (int pi = 0; pi < npairs; ++pi) {
          const int s0 = p.h_shift[2 * pi];
          const int s1 = 2 * pi + 1 < p.ntaps ? p.h_shift[2 * pi + 1] : s0 + 1;   // an odd tap out pairs with a dummy block
          const uint64_t adesc = make_sdesc(st + ATOM_BYTES + (uint32_t)s0 * ROW, (uint32_t)(s1 - s0) * ROW, SBO, 2u);
          if (ksteps == 4) {
            umma_f16_steps<4, (int)KSTEP>(tmem_base + (uint32_t)(pi * 64), adesc, bdesc, IDESC, ck > ck0 ? 1u : 0u);
          } else {
            for (int j = 0; j < ksteps; ++j)
              umma_f16(tmem_base + (uint32_t)(pi * 64), adesc + KSTEP * j, bdesc + KSTEP * j, IDESC, (ck > ck0 || j) ? 1u : 0u);
          }
        }
        umma_commit(empty_bar + s);
      }
      __syncwarp();
      if (++s == STAGES) { s = 0; par ^= 1u; }
    }
    if (elect_one()) umma_commit(tmem_full);
    __syncwarp();
  }
  __syncwarp();
  mbar_wait(tmem_full, 0);
  tc_fence_after();

  // epilogue: lane = (tap of the pair, shifted channel), columns = anchor channels
  const int m = threadIdx.x >> 6, rs = threadIdx.x & 63;
  for (int pi = 0; pi < npairs; ++pi) {
    const int t = 2 * pi + m;
    const bool valid = t < p.ntaps && ck1 > ck0;
    const int tix = valid ? p.tap_idx[t] : 0;
#pragma unroll 1
    for (int c0 = 0; c0 < 64; c0 += 32) {
      uint32_t v[32];
      tmem_ld32(tmem_base + ((uint32_t)(warp * 32) << 16) + (uint32_t)(pi * 64 + c0), v);
      if (!valid) continue;
      // consecutive lanes = consecutive shifted channels: every atomic instruction covers 128 contiguous bytes when
      // the shifted-channel stride is 1 (packed scratch)
      float* dst = p.s_rs == 1 ? p.dw + (int64_t)c0 * p.s_ra + (int64_t)tix * p.s_t + rs
                               : p.dw + ((int64_t)c0 * p.Cs + rs) * p.T + tix;
      const int64_t stride = p.s_rs == 1 ? p.s_ra : (int64_t)p.Cs * p.T;
#pragma unroll
      for (int i = 0; i < 32; ++i) atomicAdd(dst + (int64_t)i * stride, __uint_as_float(v[i]));
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 2) tmem_dealloc<512>(tmem_base);
}

// packed scratch [ra][tap][rs] -> parameter layout [ra][rs][tap] (accumulating), and re-zero the scratch.
// One CTA per (ra, RC shifted channels): float4 reads of T x RC floats, coalesced read-modify-write of RC*T floats.
// UNPACK_RA anchor rows per CTA (a CTA per row was 1152 floats of work: launch / tail bound, 4x off the HBM time).
constexpr int UNPACK_RA = 4;
template <int RC>
__global__ void __launch_bounds__(256) wgrad_unpack_kernel(float* __restrict__ scratch, float* __restrict__ dw, int Ca, int Cs, int T) {
  __shared__ float s[UNPACK_RA][BVAE_MAX_TAPS][RC + 1];
  const int ra0 = blockIdx.y * UNPACK_RA, rs0 = blockIdx.x * RC;
  const int nra = min(UNPACK_RA, Ca - ra0);
  const int per = T * (RC / 4);
  for (int e0 = threadIdx.x; e0 < nra * per; e0 += 3 * 256) {
    float4* q[3];
    float4 v[3];
#pragma unroll
    for (int u = 0; u < 3; ++u) {
      const int e = e0 + u * 256;
      q[u] = nullptr;
      if (e < nra * per) {
        const int a = e / per, e2 = e - a * per;
        const int t = e2 / (RC / 4), r = (e2 % (RC / 4)) * 4;
        q[u] = reinterpret_cast<float4*>(scratch + ((int64_t)(ra0 + a) * T + t) * Cs + rs0 + r);
        v[u] = *q[u];
      }
    }
#pragma unroll
    for (int u = 0; u < 3; ++u) {
      const int e = e0 + u * 256;
      if (!q[u]) continue;
      const int a = e / per, e2 = e - a * per;
      const int t = e2 / (RC / 4), r = (e2 % (RC / 4)) * 4;
      *q[u] = make_float4(0.f, 0.f, 0.f, 0.f);
      s[a][t][r] = v[u].x; s[a][t][r + 1] = v[u].y; s[a][t][r + 2] = v[u].z; s[a][t][r + 3] = v[u].w;
    }
  }
  __syncthreads();
  const int row = T * RC;
  const int total = nra * row;
  // read-modify-write in batches of 6 independent loads per thread (the plain loop exposed one DRAM latency per element)
  for (int e0 = threadIdx.x; e0 < total; e0 += 6 * 256) {
    float* ptr[6];
    float old[6], add[6];
#pragma unroll
    for (int u = 0; u < 6; ++u) {
      const int e = e0 + u * 256;
      ptr[u] = nullptr;
      if (e < total) {
        const int a = e / row, e2 = e - a * row;
        ptr[u] = dw + ((int64_t)(ra0 + a) * Cs + rs0) * T + e2;
        add[u] = s[a][e2 % T][e2 / T];
        old[u] = *ptr[u];
      }
    }
#pragma unroll
    for (int u = 0; u < 6; ++u)
      if (ptr[u]) *ptr[u] = old[u] + add[u];
  }
}

// ---------------------------------------------------------------------------------------------------------
// host side: tensor maps, tile selection, dispatch
// ---------------------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode() {
  static EncodeTiledFn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* f = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &f, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = (EncodeTiledFn)f;
  });
  return fn;
}

// 4-D map over a (possibly strided) NHWC view: dims {C, Wv, Hv, N}
static int make_view_map(CUtensorMap* m, const void* base, int C, int Wv, int Hv, int N, int64_t sw_elems,
                         int64_t sh_elems, int64_t sn_elems, int box_c, int bw, int bh, int bn, bool sw128) {
  EncodeTiledFn enc = get_encode();
  BVAE_REQUIRE(enc, BVAE_ERR_CUDA, "cuTensorMapEncodeTiled is not available from the driver");
  cuuint64_t dims[4] = {(cuuint64_t)C, (cuuint64_t)Wv, (cuuint64_t)Hv, (cuuint64_t)N};
  cuuint64_t strides[3] = {(cuuint64_t)sw_elems * 2, (cuuint64_t)sh_elems * 2, (cuuint64_t)sn_elems * 2};
  cuuint32_t box[4] = {(cuuint32_t)box_c, (cuuint32_t)bw, (cuuint32_t)bh, (cuuint32_t)bn};
  cuuint32_t es[4] = {1, 1, 1, 1};
  CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(base), dims, strides, box, es,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, sw128 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B,
                   CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  BVAE_REQUIRE(r == CUDA_SUCCESS, BVAE_ERR_CUDA,
               "cuTensorMapEncodeTiled(4d) failed: %d (dims %d,%d,%d,%d strides %lld,%lld,%lld box %d,%d,%d,%d)", (int)r, C, Wv,
               Hv, N, (long long)sw_elems * 2, (long long)sh_elems * 2, (long long)sn_elems * 2, box_c, bw, bh, bn);
  return BVAE_OK;
}

// 5-D map over the same view with the channel axis split into 64-channel blocks: dims {64, Wv, Hv, N, C/64}; a box
// {64, bw, bh, bn, blocks} lands as `blocks` consecutive [bn*bh*bw rows][64 ch] tiles (wgrad_tc_kernel, WT)
static int make_view_map5(CUtensorMap* m, const void* base, int C, int Wv, int Hv, int N, int64_t sw_elems, int64_t sh_elems,
                          int64_t sn_elems, int bw, int bh, int bn, int blocks) {
  EncodeTiledFn enc = get_encode();
  BVAE_REQUIRE(enc, BVAE_ERR_CUDA, "cuTensorMapEncodeTiled is not available from the driver");
  cuuint64_t dims[5] = {64, (cuuint64_t)Wv, (cuuint64_t)Hv, (cuuint64_t)N, (cuuint64_t)(C / 64)};
  cuuint64_t strides[4] = {(cuuint64_t)sw_elems * 2, (cuuint64_t)sh_elems * 2, (cuuint64_t)sn_elems * 2, 128};
  cuuint32_t box[5] = {64, (cuuint32_t)bw, (cuuint32_t)bh, (cuuint32_t)bn, (cuuint32_t)blocks};
  cuuint32_t es[5] = {1, 1, 1, 1, 1};
  CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 5, const_cast<void*>(base), dims, strides, box, es,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  BVAE_REQUIRE(r == CUDA_SUCCESS, BVAE_ERR_CUDA, "cuTensorMapEncodeTiled(5d) failed: %d (C %d dims %d,%d,%d box %d,%d,%d,%d)",
               (int)r, C, Wv, Hv, N, bw, bh, bn, blocks);
  return BVAE_OK;
}

// fp32 output view {C, Wv, Hv, N} (strides in elements), box {32 floats = 128 B of channels, bw, bh, bn}, 128B swizzle
static int make_out_map(CUtensorMap* m, const float* base, int C, int Wv, int Hv, int N, int64_t sw_elems, int64_t sh_elems,
                        int64_t sn_elems, int bw, int bh, int bn) {
  EncodeTiledFn enc = get_encode();
  BVAE_REQUIRE(enc, BVAE_ERR_CUDA, "cuTensorMapEncodeTiled is not available from the driver");
  cuuint64_t dims[4] = {(cuuint64_t)C, (cuuint64_t)Wv, (cuuint64_t)Hv, (cuuint64_t)N};
  cuuint64_t strides[3] = {(cuuint64_t)sw_elems * 4, (cuuint64_t)sh_elems * 4, (cuuint64_t)sn_elems * 4};
  cuuint32_t box[4] = {32, (cuuint32_t)bw, (cuuint32_t)bh, (cuuint32_t)bn};
  cuuint32_t es[4] = {1, 1, 1, 1};
  CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, const_cast<float*>(base), dims, strides, box, es,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  BVAE_REQUIRE(r == CUDA_SUCCESS, BVAE_ERR_CUDA, "cuTensorMapEncodeTiled(out) failed: %d (dims %d,%d,%d,%d box %d,%d,%d)",
               (int)r, C, Wv, Hv, N, bw, bh, bn);
  return BVAE_OK;
}

static int make_w_map(CUtensorMap* m, const void* base, int K, int rows, int pitch, int box_k, int box_rows, bool sw128) {
  EncodeTiledFn enc = get_encode();
  BVAE_REQUIRE(enc, BVAE_ERR_CUDA, "cuTensorMapEncodeTiled is not available from the driver");
  cuuint64_t dims[2] = {(cuuint64_t)K, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)pitch * 2};
  cuuint32_t box[2] = {(cuuint32_t)box_k, (cuuint32_t)box_rows};
  cuuint32_t es[2] = {1, 1};
  CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides, box, es,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, sw128 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B,
                   CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  BVAE_REQUIRE(r == CUDA_SUCCESS, BVAE_ERR_CUDA, "cuTensorMapEncodeTiled(2d) failed: %d (K %d rows %d pitch %d box %d,%d)",
               (int)r, K, rows, pitch, box_k, box_rows);
  return BVAE_OK;
}

static inline int floordiv(int a, int b) { return (a >= 0) ? a / b : -((-a + b - 1) / b); }

// choose the pixel box (bn, bh, bw) with bn*bh*bw <= cap that needs the fewest boxes to cover [N, QH, QW]
static void pick_box(int N, int QH, int QW, int cap, int* bw_, int* bh_, int* bn_) {
  static std::mutex mu;
  static std::unordered_map<uint64_t, uint32_t> cache;
  const uint64_t key = ((uint64_t)N << 40) | ((uint64_t)QH << 24) | ((uint64_t)QW << 8) | (uint64_t)(cap & 0xff);
  {
    std::lock_guard<std::mutex> g(mu);
    auto it = cache.find(key);
    if (it != cache.end()) {
      *bw_ = it->second & 0x3ff; *bh_ = (it->second >> 10) & 0x3ff; *bn_ = (it->second >> 20) & 0x3ff;
      return;
    }
  }
  long best = -1;
  int bbw = 1, bbh = 1, bbn = 1;
  for (int bw = 1; bw <= QW && bw <= cap; ++bw) {
    if (bw < QW && bw * 2 <= QW && (QW % bw) && bw < 8) continue;       // prune silly narrow boxes
    for (int bh = 1; bh <= QH && bh * bw <= cap; ++bh) {
      int bn = cap / (bw * bh);
      if (bn > N) bn = N;
      if (bn > 256) bn = 256;
      if (bn < 1) continue;
      if (cap == 64) {
        // weight-gradient K chunks cost one MMA per 16 pixel rows; boxes of a multiple of 16 rows qualify for the one-request-
        // per-operand loads of wgrad_tc_kernel<.., WT> and win ties (also try fewer samples per box to get there)
        for (int pass = 0; pass < 2; ++pass) {
          int b2 = bn;
          if (pass == 1) {
            while (b2 > 1 && (bw * bh * b2) % 16 != 0) --b2;
            if (b2 == bn || (bw * bh * b2) % 16 != 0) break;
          }
          const int rows = bw * bh * b2;
          const long tiles = (long)ceil_div(QW, bw) * ceil_div(QH, bh) * ceil_div(N, b2) * ceil_div(rows, 16);
          const bool m16 = rows % 16 == 0, bm16 = (bbw * bbh * bbn) % 16 == 0;
          if (best < 0 || tiles < best || (tiles == best && ((m16 && !bm16) || (m16 == bm16 && (bw > bbw || (bw == bbw && b2 < bbn)))))) {
            best = tiles; bbw = bw; bbh = bh; bbn = b2;
          }
        }
        continue;
      }
      long tiles = (long)ceil_div(QW, bw) * ceil_div(QH, bh) * ceil_div(N, bn);
      // ties: wider rows first, then boxes that stay inside one sample (needed by the fused statistics)
      if (best < 0 || tiles < best || (tiles == best && (bw > bbw || (bw == bbw && bn < bbn)))) { best = tiles; bbw = bw; bbh = bh; bbn = bn; }
    }
  }
  *bw_ = bbw; *bh_ = bbh; *bn_ = bbn;
  std::lock_guard<std::mutex> g(mu);
  cache[key] = (uint32_t)bbw | ((uint32_t)bbh << 10) | ((uint32_t)bbn << 20);
}

// Build the strided views a tap list needs.  A tap reads pixel (q*s + d): with d = s*e + f (0 <= f < s) this is
// element (q + e) of the sub-lattice f, f+s, f+2s, ... -> one tensor map per distinct (fy, fx).
struct ViewPlan {
  int nviews;
  int fy[MAX_VIEWS], fx[MAX_VIEWS];
  int tap_view[BVAE_MAX_TAPS], tap_ex[BVAE_MAX_TAPS], tap_ey[BVAE_MAX_TAPS];
};
static bool plan_views(int ntaps, const int* dy, const int* dx, int sy, int sx, ViewPlan* vp) {
  vp->nviews = 0;
  for (int t = 0; t < ntaps; ++t) {
    const int ey = floordiv(dy[t], sy), ex = floordiv(dx[t], sx);
    const int fy = dy[t] - ey * sy, fx = dx[t] - ex * sx;
    int v = -1;
    for (int i = 0; i < vp->nviews; ++i)
      if (vp->fy[i] == fy && vp->fx[i] == fx) v = i;
    if (v < 0) {
      if (vp->nviews == MAX_VIEWS) return false;
      v = vp->nviews++;
      vp->fy[v] = fy; vp->fx[v] = fx;
    }
    vp->tap_view[t] = v; vp->tap_ex[t] = ex; vp->tap_ey[t] = ey;
  }
  return true;
}

static int pick_bn(int Cout) {
  const int cands[5] = {256, 192, 128, 64, 32};
  for (int i = 0; i < 5; ++i)
    if (Cout % cands[i] == 0) return cands[i];
  return 0;
}

int conv_tc_eligible(const bvae_conv_desc* d) {
  if (d->C % 32 || d->Cout % 32 || d->x_pitch % 8 || d->y_pitch % 8 || d->w_pitch % 8) return 0;
  if (((uintptr_t)d->x | (uintptr_t)d->w) & 15) return 0;
  if ((uintptr_t)d->y & 15) return 0;
  if (d->addend && (((uintptr_t)d->addend & 15) || d->add_pitch % 8)) return 0;
  if (d->mask && (((uintptr_t)d->mask & 15) || d->mask_pitch % 8)) return 0;
  ViewPlan vp;
  if (!plan_views(d->ntaps, d->dy, d->dx, d->sy, d->sx, &vp)) return 0;
  return pick_bn(d->Cout) != 0;
}

int conv_tc_stats_ok(const bvae_conv_desc* d) {
  if (!conv_tc_eligible(d) || !d->out_f32 || d->act || d->addend || d->mask) return 0;
  int QHm = d->QH, QWm = d->QW;
  for (int i = 0; i < d->nphase; ++i) {
    if (i == 0) QHm = QWm = 0;
    if (d->ph_QH[i] > QHm) QHm = d->ph_QH[i];
    if (d->ph_QW[i] > QWm) QWm = d->ph_QW[i];
  }
  int bw, bh, bn;
  pick_box(d->N, QHm, QWm, 128, &bw, &bh, &bn);
  return bn == 1;
}

template <int KB, int BN, bool BRES>
static int launch_conv2_impl(const ConvTcParams& P, long tiles, cudaStream_t stream) {
  constexpr int B_BYTES = BN * KB * 2;
  constexpr int STAGE = BRES ? 128 * KB * 2 : 128 * KB * 2 + B_BYTES;
  constexpr int YSTAGE = BN <= 128 ? 33 * 1024 : 0;             // two output slabs of the TMA-store epilogue (+ alignment)
  constexpr int YSTAGE2 = (ConvTc2Cfg<BN>::EG - 1) * 32 * 1024; // the second epilogue group's slabs (BN <= 64)
  constexpr int BUDGET = (BRES ? 128 * 1024 : 200 * 1024) - YSTAGE;   // resident weights take up to 72 KB of their own
  constexpr int ST_RAW = BUDGET / STAGE;
  // small-channel layers are bound by the bytes in flight per SM (8 KB stages): give them a deep ring
  constexpr int STAGES = ST_RAW > 16 ? 16 : ST_RAW;
  const int smem = 1024 + (BRES ? P.ntaps * P.kchunks * B_BYTES : 0) + STAGES * STAGE + (2 * STAGES + 5) * 8 + 32 + YSTAGE + YSTAGE2;
  static int attr_smem = 0;
  static int num_sms = 148;
  if (smem > attr_smem) {
    cudaError_t e = cudaFuncSetAttribute(conv_tc2_kernel<KB, BN, STAGES, BRES>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    BVAE_REQUIRE(e == cudaSuccess, BVAE_ERR_CUDA, "conv_tc2: cudaFuncSetAttribute(%d) failed: %s", smem, cudaGetErrorString(e));
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&num_sms, cudaDevAttrMultiProcessorCount, dev);
    attr_smem = smem;
  }
  const int grid = (int)(tiles < num_sms ? tiles : num_sms);
  conv_tc2_kernel<KB, BN, STAGES, BRES><<<grid, ConvTc2Cfg<BN>::THREADS, smem, stream>>>(P);
  note_kernel("conv_tc2_kernel<%d,%d,%d,%d>%s", KB, BN, STAGES, (int)BRES, P.halo ? "+halo" : "");
  return check_launch("conv_tc2");
}

template <int KB, int BN>
static int launch_conv2(const ConvTcParams& P, long tiles, cudaStream_t stream) {
  // weights resident in shared memory when one N tile covers Cout and all taps fit in 96 KB
  const bool bres = P.n_tiles == 1 && (long)P.ntaps * P.kchunks * (BN * KB * 2) <= 72 * 1024 && tiles >= 2 * 148;
  return bres ? launch_conv2_impl<KB, BN, true>(P, tiles, stream) : launch_conv2_impl<KB, BN, false>(P, tiles, stream);
}

// Halo mode applies to single-phase stride-1 layers whose weights stay resident (see launch_conv2): the output tile is
// RH image rows of the PADDED width PW = QW + (dx_max - dx_min), flattened, so that tap (dy, dx) is the same smem tile
// shifted by (dy - dy_min) * PW + (dx - dx_min) rows.  Output rows that fall on padding columns are discarded.
static int plan_halo(const bvae_conv_desc* d, ConvTcParams* P, int KB, int BN) {
  if (KB != 64 || P->nphase != 1 || d->sy != 1 || d->sx != 1 || d->osy != 1 || d->osx != 1 ||
      P->n_tiles != 1 || d->ntaps < 4 || d->stats)
    return BVAE_OK;
  if ((long)d->ntaps * P->kchunks * (BN * KB * 2) > 72 * 1024) return BVAE_OK;
  int dy0 = d->dy[0], dy1 = d->dy[0], dx0 = d->dx[0], dx1 = d->dx[0];
  for (int t = 1; t < d->ntaps; ++t) {
    dy0 = d->dy[t] < dy0 ? d->dy[t] : dy0; dy1 = d->dy[t] > dy1 ? d->dy[t] : dy1;
    dx0 = d->dx[t] < dx0 ? d->dx[t] : dx0; dx1 = d->dx[t] > dx1 ? d->dx[t] : dx1;
  }
  const int QH = P->ph_QH[0], QW = P->ph_QW[0];
  const int PW = QW + (dx1 - dx0);
  if (PW > 128) return BVAE_OK;
  int RH = 128 / PW;
  if (RH > QH) RH = QH;
  const int rows = (RH + dy1 - dy0) * PW;
  int reach = 128 + (dy1 - dy0) * PW + (dx1 - dx0);          // rows the shifted descriptors can touch
  if (reach < rows) reach = rows;
  const int stage = ((reach * 128 + 1023) / 1024) * 1024;
  const long tiles = (long)d->N * ceil_div(QH, RH);
  if (RH + dy1 - dy0 > 256 || QW * RH * 10 < 128 * 8 || stage > 40 * 1024 || tiles < 2 * 148) return BVAE_OK;
  int rc = make_view_map(&P->amap[0], d->x, d->C, d->W, d->H, d->N, d->x_pitch, (int64_t)d->W * d->x_pitch,
                         (int64_t)d->H * d->W * d->x_pitch, KB, PW, RH + dy1 - dy0, 1, true);
  if (rc) return rc;
  P->halo = 1;
  P->halo_x0 = dx0; P->halo_y0 = dy0; P->halo_rows = rows; P->halo_stage = stage;
  P->halo_stages = (80 * 1024) / stage;                      // the BRES ring region: 5 stages of 16 KB (launch_conv2_impl)
  for (int t = 0; t < d->ntaps; ++t) P->halo_shift[t] = (d->dy[t] - dy0) * PW + (d->dx[t] - dx0);
  P->bw = PW; P->bh = RH; P->bn = 1;
  P->tiles_w = 1; P->tiles_h = ceil_div(QH, RH); P->tiles_n = d->N;
  return BVAE_OK;
}

int conv_tc_launch(const bvae_conv_desc* d, cudaStream_t stream) {
  ConvTcParams P;
  memset(&P, 0, sizeof(P));
  const bool sw128 = (d->C % 64 == 0);
  const int KB = sw128 ? 64 : 32;
  const int BN = pick_bn(d->Cout);
  ViewPlan vp;
  BVAE_REQUIRE(plan_views(d->ntaps, d->dy, d->dx, d->sy, d->sx, &vp), BVAE_ERR_UNSUPPORTED, "conv_tc: too many views");
  int QHm = d->QH, QWm = d->QW;
  if (d->nphase > 0) {
    QHm = QWm = 0;
    int t0 = 0;
    P.nphase = d->nphase;
    for (int i = 0; i < d->nphase; ++i) {
      P.ph_tap0[i] = t0; P.ph_ntaps[i] = d->ph_ntaps[i]; P.ph_ooy[i] = d->ph_ooy[i]; P.ph_oox[i] = d->ph_oox[i];
      P.ph_QH[i] = d->ph_QH[i]; P.ph_QW[i] = d->ph_QW[i];
      t0 += d->ph_ntaps[i];
      if (d->ph_QH[i] > QHm) QHm = d->ph_QH[i];
      if (d->ph_QW[i] > QWm) QWm = d->ph_QW[i];
    }
    BVAE_REQUIRE(t0 == d->ntaps, BVAE_ERR_SHAPE, "conv_tc: phase tap counts do not add up to ntaps");
  } else {
    P.nphase = 1;
    P.ph_tap0[0] = 0; P.ph_ntaps[0] = d->ntaps; P.ph_ooy[0] = d->ooy; P.ph_oox[0] = d->oox;
    P.ph_QH[0] = d->QH; P.ph_QW[0] = d->QW;
  }
  pick_box(d->N, QHm, QWm, 128, &P.bw, &P.bh, &P.bn);
  for (int v = 0; v < vp.nviews; ++v) {
    const int Hv = ceil_div(d->H - vp.fy[v], d->sy), Wv = ceil_div(d->W - vp.fx[v], d->sx);
    BVAE_REQUIRE(Hv > 0 && Wv > 0, BVAE_ERR_SHAPE, "conv_tc: empty view");
    const bf16* base = (const bf16*)d->x + ((int64_t)vp.fy[v] * d->W + vp.fx[v]) * d->x_pitch;
    int rc = make_view_map(&P.amap[v], base, d->C, Wv, Hv, d->N, (int64_t)d->sx * d->x_pitch,
                           (int64_t)d->sy * d->W * d->x_pitch, (int64_t)d->H * d->W * d->x_pitch, KB, P.bw, P.bh, P.bn, sw128);
    if (rc) return rc;
  }
  int rc = make_w_map(&P.bmap, d->w, d->ntaps * d->C, d->Cout, d->w_pitch, KB, BN, sw128);
  if (rc) return rc;
  for (int t = 0; t < d->ntaps; ++t) { P.tap_view[t] = vp.tap_view[t]; P.tap_ex[t] = vp.tap_ex[t]; P.tap_ey[t] = vp.tap_ey[t]; }
  P.ntaps = d->ntaps; P.kchunks = d->C / KB; P.C = d->C;
  P.tiles_w = ceil_div(QWm, P.bw); P.tiles_h = ceil_div(QHm, P.bh); P.tiles_n = ceil_div(d->N, P.bn);
  P.n_tiles = d->Cout / BN;
  P.N = d->N; P.QH = QHm; P.QW = QWm; P.Cout = d->Cout;
  P.y = d->y; P.bias = d->bias; P.addend = d->addend; P.mask = d->mask; P.stats = d->stats;
  P.OH = d->OH; P.OW = d->OW; P.y_pitch = d->y_pitch; P.osy = d->osy; P.osx = d->osx; P.ooy = d->ooy; P.oox = d->oox;
  P.add_pitch = d->add_pitch; P.mask_pitch = d->mask_pitch; P.act = d->act; P.out_f32 = d->out_f32;
  P.slope = d->slope; P.mask_slope = d->mask_slope;
  rc = plan_halo(d, &P, KB, BN);
  if (rc) return rc;
  // TMA-store epilogue for fp32 outputs only: on the bf16 data gradients it measured slower (0.79 vs 0.65 ms on 64->64 3x3,
  // the mask rows are already prefetched there and the extra barriers cost more than the store requests save)
  if (d->out_f32 && !d->stats && BN <= 128 && d->y_pitch % 4 == 0 && ((uintptr_t)d->y & 15) == 0) {
    for (int i = 0; i < P.nphase; ++i) {
      const float* base = (const float*)d->y + ((int64_t)P.ph_ooy[i] * d->OW + P.ph_oox[i]) * d->y_pitch;
      rc = make_out_map(&P.ymap[i], base, d->Cout, P.ph_QW[i], P.ph_QH[i], d->N, (int64_t)d->osx * d->y_pitch,
                        (int64_t)d->osy * d->OW * d->y_pitch, (int64_t)d->OH * d->OW * d->y_pitch, P.bw, P.bh, P.bn);
      if (rc) return rc;
    }
    P.tma_store = 1;
  }
  const long grid = (long)P.tiles_w * P.tiles_h * P.tiles_n * P.n_tiles * P.nphase;
  BVAE_REQUIRE(grid > 0 && grid < (1l << 31), BVAE_ERR_SHAPE, "conv_tc: grid too large");
#define CONV2_CASE(kb, bn) if (KB == kb && BN == bn) return launch_conv2<kb, bn>(P, grid, stream)
  CONV2_CASE(64, 256); CONV2_CASE(64, 192); CONV2_CASE(64, 128); CONV2_CASE(64, 64); CONV2_CASE(64, 32);
  CONV2_CASE(32, 256); CONV2_CASE(32, 192); CONV2_CASE(32, 128); CONV2_CASE(32, 64); CONV2_CASE(32, 32);
#undef CONV2_CASE
  set_error("conv_tc: no kernel for KB=%d BN=%d", KB, BN);
  return BVAE_ERR_UNSUPPORTED;
}

int wgrad_tc_eligible(const bvae_wgrad_desc* d) {
  if (d->Ca % 32 || d->Cs % 32 || d->a_pitch % 8 || d->s_pitch % 8) return 0;
  if (d->Ca > 128 && d->Ca % 128) return 0;
  if (((uintptr_t)d->a | (uintptr_t)d->s) & 15) return 0;
  ViewPlan vp;
  return plan_views(d->ntaps, d->dy, d->dx, d->sy, d->sx, &vp) ? 1 : 0;
}

constexpr int WT_RING_BUDGET = 200 * 1024;     // shared memory the WT ring may take (+ 2 KB of alignment / barriers)
template <int NS, int STAGES>
static int launch_wgrad_wt(const WgradTcParams& P, int grid, cudaStream_t stream) {
  const int smem = 1024 + 1024 + P.wt_stages * P.wt_stage_bytes;
  static bool attr_done = false;
  if (!attr_done) {
    cudaError_t e = cudaFuncSetAttribute(wgrad_tc_kernel<64, NS, STAGES, true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         WT_RING_BUDGET + 2048);
    BVAE_REQUIRE(e == cudaSuccess, BVAE_ERR_CUDA, "wgrad_tc: cudaFuncSetAttribute failed: %s", cudaGetErrorString(e));
    attr_done = true;
  }
  wgrad_tc_kernel<64, NS, STAGES, true><<<grid, 128, smem, stream>>>(P);
  note_kernel("wgrad_tc_kernel<64,%d,%d>+wt", NS, P.wt_stages);
  return check_launch("wgrad_tc");
}

template <int CB, int NS, int STAGES>
static int launch_wgrad(const WgradTcParams& P, int grid, cudaStream_t stream) {
  constexpr int max_tpc = (512 / NS) > BVAE_MAX_TAPS ? BVAE_MAX_TAPS : (512 / NS);
  constexpr int smem = 1024 + STAGES * (128 / CB + max_tpc * (NS / CB)) * (64 * CB * 2) + (2 * STAGES + 1) * 8 + 16;
  static bool attr_done = false;
  if (!attr_done) {
    cudaError_t e = cudaFuncSetAttribute(wgrad_tc_kernel<CB, NS, STAGES>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    BVAE_REQUIRE(e == cudaSuccess, BVAE_ERR_CUDA, "wgrad_tc: cudaFuncSetAttribute(%d) failed: %s", smem, cudaGetErrorString(e));
    attr_done = true;
  }
  if (P.wt == 1) {
    if constexpr (CB == 64) return launch_wgrad_wt<NS, STAGES>(P, grid, stream);
  }
  wgrad_tc_kernel<CB, NS, STAGES><<<grid, 128, smem, stream>>>(P);
  note_kernel("wgrad_tc_kernel<%d,%d,%d>", CB, NS, STAGES);
  return check_launch("wgrad_tc");
}

// acc_cols = accumulator columns a CTA drains in its epilogue (0: the halo kernel, which keeps the fill heuristic)
static void wgrad_finish(const bvae_wgrad_desc* d, WgradTcParams* P, int out_tiles, bool* packed_, int acc_cols = 0) {
  const int max_splits = ceil_div(P->nchunks, 8);
  int splits = 1;
  if (acc_cols > 0) {
    // Pixel splits from a cost model (round 3).  ncu on 512->512 3x3 at 6x4 x 512 bars (40 output tiles x 7 splits = 280 CTAs,
    // 28 chunks each, 85 us): a CTA spends only ~55 % of its 42 us in the K loop (0.8 us per 64-pixel chunk); zeroing the
    // ring, TMEM allocation, the pipeline fill and above all the epilogue -- 128 x 512 fp32 as vector atomics, not overlapped
    // with anything because the tile owns all of TMEM -- are a fixed ~24 chunk-equivalents, paid once per WAVE.  The old rule
    // (fill ~2 waves) bought its fill with a second round of fixed costs and 2-3x the atomic traffic.
    const double fixed = 8.0 + 16.0 * (double)acc_cols / 512.0;
    double best = 1e30;
    for (int sp = 1; sp <= max_splits && sp <= 128; ++sp) {
      const int cps = ceil_div(P->nchunks, sp), rsp = ceil_div(P->nchunks, cps);
      const long ctas = (long)out_tiles * rsp, waves = (ctas + 147) / 148;
      const double cost = (double)waves * (fixed + (double)cps);
      if (cost < best - 1e-9) { best = cost; splits = rsp; }
    }
  } else {
    // aim at ~2 waves of 148 CTAs and pick the candidate that fills its last wave best
    const int centre = ceil_div(148 * 2, out_tiles);
    double best_fill = -1.0;
    for (int sp = (centre > 3 ? centre - 2 : 1); sp <= centre + 2; ++sp) {
      if (sp > max_splits) break;
      const long ctas = (long)out_tiles * sp;
      const long waves = (ctas + 147) / 148;
      const double fill = (double)ctas / (double)(waves * 148);
      if (fill > best_fill + 1e-9) { best_fill = fill; splits = sp; }
    }
  }
  if (deterministic()) splits = 1;        // one CTA accumulates a whole output tile: one ordered addition per element
  P->chunks_per_split = ceil_div(P->nchunks, splits);
  P->splits = ceil_div(P->nchunks, P->chunks_per_split);
  // Reduction target.  Many pixel splits over a small weight (encoder front, decoder back): vector atomics into the
  // packed scratch, then one unpack pass.  Few splits over a large weight: scalar atomics straight into dw are cheaper
  // than an extra pass over the weight.
  const bool packed = d->T > 1 && d->scratch != nullptr && P->splits >= 3;
  if (d->T == 1) { P->dw = d->dw; P->s_ra = d->Cs; P->s_t = 0; P->s_rs = 1; }
  else if (packed) { P->dw = d->scratch; P->s_ra = (long long)d->T * d->Cs; P->s_t = d->Cs; P->s_rs = 1; }
  else { P->dw = d->dw; P->s_ra = 0; P->s_t = 0; P->s_rs = d->T; }
  *packed_ = packed;
}

static int wgrad_unpack(const bvae_wgrad_desc* d, cudaStream_t stream) {
  if (d->Cs % 128 == 0) {
    dim3 ug(d->Cs / 128, ceil_div(d->Ca, UNPACK_RA));
    wgrad_unpack_kernel<128><<<ug, 256, 0, stream>>>(d->scratch, d->dw, d->Ca, d->Cs, d->T);
  } else {
    dim3 ug(d->Cs / 32, ceil_div(d->Ca, UNPACK_RA));
    wgrad_unpack_kernel<32><<<ug, 256, 0, stream>>>(d->scratch, d->dw, d->Ca, d->Cs, d->T);
  }
  return check_launch("wgrad_unpack");
}

static int wgrad_halo_try(const bvae_wgrad_desc* d, const ViewPlan* vp, cudaStream_t stream, int* done) {
  *done = 0;
  if (d->Ca != 64 || d->Cs != 64 || d->sy != 1 || d->sx != 1 || d->ntaps < 4 || d->ntaps > 16 || vp->nviews != 1)
    return BVAE_OK;
  int dy0 = d->dy[0], dy1 = d->dy[0], dx0 = d->dx[0], dx1 = d->dx[0];
  for (int t = 1; t < d->ntaps; ++t) {
    dy0 = d->dy[t] < dy0 ? d->dy[t] : dy0; dy1 = d->dy[t] > dy1 ? d->dy[t] : dy1;
    dx0 = d->dx[t] < dx0 ? d->dx[t] : dx0; dx1 = d->dx[t] > dx1 ? d->dx[t] : dx1;
  }
  const int PW = d->AW + (dx1 - dx0);
  if (PW > 64) return BVAE_OK;
  int RH = 64 / PW;
  if (RH > d->AH) RH = d->AH;
  if (d->AW * RH * 4 < 64 * 3) return BVAE_OK;                  // < 75 % of the contraction rows would be real pixels
  WgradTcParams P;
  memset(&P, 0, sizeof(P));
  P.h_PW = PW; P.h_RH = RH; P.h_rows_a = RH * PW; P.h_rows_s = (RH + dy1 - dy0) * PW;
  P.h_x0 = dx0; P.h_y0 = dy0;
  int reach = 64 + (dy1 - dy0) * PW + (dx1 - dx0) + 1;          // rows the shifted descriptors can touch
  if (reach < P.h_rows_s) reach = P.h_rows_s;
  P.h_stage = 64 * 128 + ((reach * 128 + 1023) / 1024) * 1024;
  P.h_stages = (190 * 1024) / P.h_stage;
  if (P.h_stages > 8) P.h_stages = 8;
  if (P.h_stages < 2) return BVAE_OK;
  int rc = make_view_map(&P.amap, d->a, d->Ca, d->AW, d->AH, d->N, d->a_pitch, (int64_t)d->AW * d->a_pitch,
                         (int64_t)d->AH * d->AW * d->a_pitch, 64, PW, RH, 1, true);
  if (rc) return rc;
  rc = make_view_map(&P.smap[0], d->s, d->Cs, d->SW, d->SH, d->N, d->s_pitch, (int64_t)d->SW * d->s_pitch,
                     (int64_t)d->SH * d->SW * d->s_pitch, 64, PW, RH + dy1 - dy0, 1, true);
  if (rc) return rc;
  // taps in ascending shift order (the second block of a pair lies behind the first)
  int order[BVAE_MAX_TAPS];
  for (int t = 0; t < d->ntaps; ++t) order[t] = t;
  for (int i = 1; i < d->ntaps; ++i)
    for (int k = i; k > 0; --k) {
      const int a = order[k - 1], b = order[k];
      const int sa_ = (d->dy[a] - dy0) * PW + (d->dx[a] - dx0), sb_ = (d->dy[b] - dy0) * PW + (d->dx[b] - dx0);
      if (sa_ <= sb_) break;
      order[k - 1] = b; order[k] = a;
    }
  for (int t = 0; t < d->ntaps; ++t) {
    const int o = order[t];
    P.h_shift[t] = (d->dy[o] - dy0) * PW + (d->dx[o] - dx0);
    P.tap_idx[t] = d->tap_idx[o];
  }
  P.ntaps = d->ntaps; P.T = d->T;
  P.tap_groups = 1; P.tpc = d->ntaps;
  P.h_tiles_h = ceil_div(d->AH, RH);
  P.nchunks = d->N * P.h_tiles_h;
  P.Ca = d->Ca; P.Cs = d->Cs;
  bool packed = false;
  wgrad_finish(d, &P, 2, &packed);                              // one CTA per SM (it owns all 512 TMEM columns): ~148 splits
  const long grid = P.splits;
  const int smem = 1024 + P.h_stages * P.h_stage + (2 * P.h_stages + 1) * 8 + 16;
  static int attr_smem = 0;
  if (smem > attr_smem) {
    cudaError_t e = cudaFuncSetAttribute(wgrad_halo_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    BVAE_REQUIRE(e == cudaSuccess, BVAE_ERR_CUDA, "wgrad_halo: cudaFuncSetAttribute(%d) failed: %s", smem, cudaGetErrorString(e));
    attr_smem = smem;
  }
  wgrad_halo_kernel<<<(int)grid, 128, smem, stream>>>(P);
  note_kernel("wgrad_halo_kernel");
  rc = check_launch("wgrad_halo");
  *done = 1;
  if (rc || !packed) return rc;
  return wgrad_unpack(d, stream);
}

int wgrad_tc_launch(const bvae_wgrad_desc* d, cudaStream_t stream) {
  WgradTcParams P;
  memset(&P, 0, sizeof(P));
  ViewPlan vp;
  BVAE_REQUIRE(plan_views(d->ntaps, d->dy, d->dx, d->sy, d->sx, &vp), BVAE_ERR_UNSUPPORTED, "wgrad_tc: too many views");
  const bool sw128 = (d->Ca % 64 == 0) && (d->Cs % 64 == 0);
  const int CB = sw128 ? 64 : 32;
  const int NS = sw128 ? (d->Cs % 256 == 0 ? 256 : (d->Cs % 128 == 0 ? 128 : 64)) : (d->Cs % 64 == 0 ? 64 : 32);
  {
    int done = 0;
    const int rc = wgrad_halo_try(d, &vp, stream, &done);
    if (rc || done) return rc;
  }
  pick_box(d->N, d->AH, d->AW, 64, &P.bw, &P.bh, &P.bn);
  // one 5-D TMA request per operand and tap (see wgrad_tc_kernel, WT)
  const bool wt = CB == 64 && (P.bw * P.bh * P.bn) % 16 == 0;
  P.wt = wt ? 1 : 0;
  const int a_atoms = d->Ca >= 128 ? 128 / CB : d->Ca / CB;
  int rc = wt ? make_view_map5(&P.amap, d->a, d->Ca, d->AW, d->AH, d->N, d->a_pitch, (int64_t)d->AW * d->a_pitch,
                               (int64_t)d->AH * d->AW * d->a_pitch, P.bw, P.bh, P.bn, a_atoms)
              : make_view_map(&P.amap, d->a, d->Ca, d->AW, d->AH, d->N, d->a_pitch, (int64_t)d->AW * d->a_pitch,
                              (int64_t)d->AH * d->AW * d->a_pitch, CB, P.bw, P.bh, P.bn, sw128);
  if (rc) return rc;
  for (int v = 0; v < vp.nviews; ++v) {
    const int Hv = ceil_div(d->SH - vp.fy[v], d->sy), Wv = ceil_div(d->SW - vp.fx[v], d->sx);
    BVAE_REQUIRE(Hv > 0 && Wv > 0, BVAE_ERR_SHAPE, "wgrad_tc: empty view");
    const bf16* base = (const bf16*)d->s + ((int64_t)vp.fy[v] * d->SW + vp.fx[v]) * d->s_pitch;
    rc = wt ? make_view_map5(&P.smap[v], base, d->Cs, Wv, Hv, d->N, (int64_t)d->sx * d->s_pitch,
                             (int64_t)d->sy * d->SW * d->s_pitch, (int64_t)d->SH * d->SW * d->s_pitch, P.bw, P.bh, P.bn, NS / 64)
            : make_view_map(&P.smap[v], base, d->Cs, Wv, Hv, d->N, (int64_t)d->sx * d->s_pitch,
                            (int64_t)d->sy * d->SW * d->s_pitch, (int64_t)d->SH * d->SW * d->s_pitch, CB, P.bw, P.bh, P.bn, sw128);
    if (rc) return rc;
  }
  for (int t = 0; t < d->ntaps; ++t) {
    P.tap_view[t] = vp.tap_view[t]; P.tap_ex[t] = vp.tap_ex[t]; P.tap_ey[t] = vp.tap_ey[t]; P.tap_idx[t] = d->tap_idx[t];
  }
  P.ntaps = d->ntaps; P.T = d->T;
  const int max_tpc = (512 / NS) > BVAE_MAX_TAPS ? BVAE_MAX_TAPS : (512 / NS);
  if (wt) {
    P.wt_stage_bytes = (128 / 64 + max_tpc * (NS / 64)) * (P.bw * P.bh * P.bn) * 128;
    const int nst = WT_RING_BUDGET / P.wt_stage_bytes;
    P.wt_stages = nst > 4 ? 4 : (nst < 2 ? 2 : nst);
  }
  P.tap_groups = ceil_div(d->ntaps, max_tpc);
  P.tpc = ceil_div(d->ntaps, P.tap_groups);
  P.chunks_w = ceil_div(d->AW, P.bw); P.chunks_h = ceil_div(d->AH, P.bh); P.chunks_n = ceil_div(d->N, P.bn);
  P.nchunks = P.chunks_w * P.chunks_h * P.chunks_n;
  P.ra_tiles = ceil_div(d->Ca, 128); P.rs_tiles = d->Cs / NS;
  P.a_atoms = d->Ca >= 128 ? 128 / CB : d->Ca / CB;
  P.Ca = d->Ca; P.Cs = d->Cs;

  const int out_tiles = P.ra_tiles * P.rs_tiles * P.tap_groups;
  bool packed = false;
  // (the 32-channel stem layers are HBM bound and want the bytes in flight of ~2 waves: 0.84 -> 0.93 ms with the cost model)
  wgrad_finish(d, &P, out_tiles, &packed, CB == 64 ? P.tpc * NS : 0);
  const long grid = (long)out_tiles * P.splits;
  BVAE_REQUIRE(grid > 0 && grid < (1l << 31), BVAE_ERR_SHAPE, "wgrad_tc: grid too large");
  if (CB == 32) rc = NS == 64 ? launch_wgrad<32, 64, 2>(P, (int)grid, stream) : launch_wgrad<32, 32, 2>(P, (int)grid, stream);
  else if (NS == 256) rc = launch_wgrad<64, 256, 2>(P, (int)grid, stream);
  else if (NS == 128) rc = launch_wgrad<64, 128, 2>(P, (int)grid, stream);
  else rc = launch_wgrad<64, 64, 2>(P, (int)grid, stream);
  if (rc || !packed) return rc;
  return wgrad_unpack(d, stream);
}

}  // namespace bvae
