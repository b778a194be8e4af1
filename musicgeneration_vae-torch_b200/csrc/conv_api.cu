// conv_api.cu -- validation + dispatch of the contraction entry points (SIMT checker vs tcgen05 kernels).
#include "common.cuh"

namespace bvae {
int conv_simt_launch(const bvae_conv_desc* d, cudaStream_t stream);
int wgrad_simt_launch(const bvae_wgrad_desc* d, cudaStream_t stream);
int conv_tc_eligible(const bvae_conv_desc* d);
int conv_tc_launch(const bvae_conv_desc* d, cudaStream_t stream);
int conv_tc_stats_ok(const bvae_conv_desc* d);
int wgrad_tc_eligible(const bvae_wgrad_desc* d);
int wgrad_tc_launch(const bvae_wgrad_desc* d, cudaStream_t stream);
int stem_fwd_eligible(const bvae_conv_desc* d);
int stem_fwd_launch(const bvae_conv_desc* d, cudaStream_t stream);
int stem_wgrad_eligible(const bvae_wgrad_desc* d);
int stem_wgrad_launch(const bvae_wgrad_desc* d, cudaStream_t stream);
int conv_small_eligible(const bvae_conv_desc* d);
int conv_small_launch(const bvae_conv_desc* d, cudaStream_t stream);
int wgrad_small_eligible(const bvae_wgrad_desc* d);
int wgrad_small_launch(const bvae_wgrad_desc* d, cudaStream_t stream);
}  // namespace bvae

using namespace bvae;

// phase i of a multi-phase descriptor as a stand-alone single-phase descriptor
static bvae_conv_desc single_phase(const bvae_conv_desc* d, int i) {
  bvae_conv_desc s = *d;
  int t0 = 0;
  for (int k = 0; k < i; ++k) t0 += d->ph_ntaps[k];
  s.nphase = 0;
  s.ntaps = d->ph_ntaps[i];
  for (int t = 0; t < s.ntaps; ++t) { s.dy[t] = d->dy[t0 + t]; s.dx[t] = d->dx[t0 + t]; }
  s.w = (const char*)d->w + (size_t)t0 * d->C * 2;
  s.QH = d->ph_QH[i]; s.QW = d->ph_QW[i]; s.ooy = d->ph_ooy[i]; s.oox = d->ph_oox[i];
  return s;
}

extern "C" int bvae_conv_gemm(const bvae_conv_desc* d, int impl, void* stream) {
  BVAE_REQUIRE(d && d->x && d->w && d->y, BVAE_ERR_SHAPE, "conv_gemm: null pointer");
  if (d->nphase > 0) {
    BVAE_REQUIRE(d->nphase <= BVAE_MAX_PHASES, BVAE_ERR_SHAPE, "conv_gemm: nphase=%d", d->nphase);
    if (!(impl != BVAE_IMPL_SIMT && conv_tc_eligible(d))) {
      for (int i = 0; i < d->nphase; ++i) {          // kernels that take one phase at a time
        if (d->ph_QH[i] <= 0 || d->ph_QW[i] <= 0) continue;
        const bvae_conv_desc s = single_phase(d, i);
        const int rc = bvae_conv_gemm(&s, impl, stream);
        if (rc) return rc;
      }
      return BVAE_OK;
    }
    BVAE_REQUIRE(d->ntaps >= 1 && d->ntaps <= BVAE_MAX_TAPS, BVAE_ERR_SHAPE, "conv_gemm: ntaps=%d", d->ntaps);
    // the same bounds the single-phase path checks below, per phase
    BVAE_REQUIRE(d->N > 0 && d->C > 0 && d->Cout > 0, BVAE_ERR_SHAPE, "conv_gemm: empty problem");
    BVAE_REQUIRE(d->sy >= 1 && d->sx >= 1 && d->osy >= 1 && d->osx >= 1, BVAE_ERR_SHAPE, "conv_gemm: bad strides");
    BVAE_REQUIRE(d->w_pitch >= d->ntaps * d->C, BVAE_ERR_SHAPE, "conv_gemm: w_pitch too small");
    for (int i = 0; i < d->nphase; ++i) {
      BVAE_REQUIRE(d->ph_ntaps[i] >= 1 && d->ph_QH[i] >= 0 && d->ph_QW[i] >= 0, BVAE_ERR_SHAPE, "conv_gemm: bad phase %d", i);
      if (d->ph_QH[i] == 0 || d->ph_QW[i] == 0) continue;
      BVAE_REQUIRE((d->ph_QH[i] - 1) * d->osy + d->ph_ooy[i] < d->OH && (d->ph_QW[i] - 1) * d->osx + d->ph_oox[i] < d->OW,
                   BVAE_ERR_SHAPE, "conv_gemm: grid of phase %d exceeds the output tensor", i);
    }
    return conv_tc_launch(d, (cudaStream_t)stream);
  }
  BVAE_REQUIRE(d->ntaps >= 1 && d->ntaps <= BVAE_MAX_TAPS, BVAE_ERR_SHAPE, "conv_gemm: ntaps=%d", d->ntaps);
  BVAE_REQUIRE(d->N > 0 && d->QH > 0 && d->QW > 0 && d->C > 0 && d->Cout > 0, BVAE_ERR_SHAPE, "conv_gemm: empty problem");
  BVAE_REQUIRE(d->sy >= 1 && d->sx >= 1 && d->osy >= 1 && d->osx >= 1, BVAE_ERR_SHAPE, "conv_gemm: bad strides");
  BVAE_REQUIRE((d->QH - 1) * d->osy + d->ooy < d->OH && (d->QW - 1) * d->osx + d->oox < d->OW, BVAE_ERR_SHAPE,
               "conv_gemm: phase grid exceeds the output tensor");
  BVAE_REQUIRE(d->w_pitch >= d->ntaps * d->C, BVAE_ERR_SHAPE, "conv_gemm: w_pitch too small");
  BVAE_REQUIRE(!d->stats || (impl != BVAE_IMPL_SIMT && conv_tc_stats_ok(d)), BVAE_ERR_UNSUPPORTED,
               "conv_gemm: statistics fusion is not available for this problem (check bvae_conv_stats_ok)");
  if (impl == BVAE_IMPL_SIMT) return conv_simt_launch(d, (cudaStream_t)stream);
  if (impl == BVAE_IMPL_AUTO && stem_fwd_eligible(d)) return stem_fwd_launch(d, (cudaStream_t)stream);
  if (impl == BVAE_IMPL_AUTO && conv_small_eligible(d)) return conv_small_launch(d, (cudaStream_t)stream);
  const int ok = conv_tc_eligible(d);
  if (impl == BVAE_IMPL_TC) {
    BVAE_REQUIRE(ok, BVAE_ERR_UNSUPPORTED, "conv_gemm: shape not eligible for the tcgen05 kernel (C=%d Cout=%d)", d->C, d->Cout);
    return conv_tc_launch(d, (cudaStream_t)stream);
  }
  return ok ? conv_tc_launch(d, (cudaStream_t)stream) : conv_simt_launch(d, (cudaStream_t)stream);
}

extern "C" int bvae_conv_stats_ok(const bvae_conv_desc* d) {
  if (!d) return 0;
  if (d->nphase > 0) {
    if (conv_tc_eligible(d)) return conv_tc_stats_ok(d);
    for (int i = 0; i < d->nphase; ++i) {
      if (d->ph_QH[i] <= 0 || d->ph_QW[i] <= 0) continue;
      const bvae_conv_desc s = single_phase(d, i);
      if (!conv_tc_stats_ok(&s)) return 0;
    }
    return 1;
  }
  return conv_tc_stats_ok(d);
}

extern "C" int bvae_wgrad_gemm(const bvae_wgrad_desc* d, int impl, void* stream) {
  BVAE_REQUIRE(d && d->a && d->s && d->dw, BVAE_ERR_SHAPE, "wgrad_gemm: null pointer");
  BVAE_REQUIRE(d->ntaps >= 1 && d->ntaps <= BVAE_MAX_TAPS && d->T >= d->ntaps, BVAE_ERR_SHAPE, "wgrad_gemm: ntaps=%d T=%d", d->ntaps, d->T);
  BVAE_REQUIRE(d->N > 0 && d->AH > 0 && d->AW > 0 && d->Ca > 0 && d->Cs > 0, BVAE_ERR_SHAPE, "wgrad_gemm: empty problem");
  if (impl == BVAE_IMPL_SIMT) return wgrad_simt_launch(d, (cudaStream_t)stream);
  if (impl == BVAE_IMPL_AUTO && stem_wgrad_eligible(d)) return stem_wgrad_launch(d, (cudaStream_t)stream);
  if (impl == BVAE_IMPL_AUTO && wgrad_small_eligible(d)) return wgrad_small_launch(d, (cudaStream_t)stream);
  const int ok = wgrad_tc_eligible(d);
  if (impl == BVAE_IMPL_TC) {
    BVAE_REQUIRE(ok, BVAE_ERR_UNSUPPORTED, "wgrad_gemm: shape not eligible for the tcgen05 kernel (Ca=%d Cs=%d)", d->Ca, d->Cs);
    return wgrad_tc_launch(d, (cudaStream_t)stream);
  }
  return ok ? wgrad_tc_launch(d, (cudaStream_t)stream) : wgrad_simt_launch(d, (cudaStream_t)stream);
}
