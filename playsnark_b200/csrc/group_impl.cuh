// Definitions of GroupOps<F> (group_ops.cuh): the MSM pipeline, point (de)serialisation and the
// setup-side kernels for one group.  Included only by group_g1.cu / group_g2.cu, which instantiate it.
#pragma once
#include "codec.cuh"
#include "msm.cuh"

namespace ps {

// ---- setup-side kernels ---------------------------------------------------------------------------
template <class F> PS_DEV Affine<F> generator();
template <> PS_DEV Affine<Fp> generator<Fp>() {
  return Affine<Fp>{Fp::from_const<FpParams::G1X>(), Fp::from_const<FpParams::G1Y>()};
}
template <> PS_DEV Affine<Fp2> generator<Fp2>() {
  return Affine<Fp2>{Fp2{Fp::from_const<FpParams::G2X0>(), Fp::from_const<FpParams::G2X1>()},
                     Fp2{Fp::from_const<FpParams::G2Y0>(), Fp::from_const<FpParams::G2Y1>()}};
}

// table[w*255 + d-1] = d * 2^(8w) * generator, w < 32, 1 <= d <= 255
template <class F>
struct FixedBaseTableK {
  static constexpr int BLOCK = 64;
  PS_DEV static void run(uint32_t tid, Affine<F>* table) {
    uint32_t w = tid / 255, d = tid % 255 + 1;
    uint32_t k[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    k[w / 4] = d << (8 * (w % 4));
    XYZZ<F> r = xyzz_scalar_mul(XYZZ<F>::from_affine(generator<F>()), k, 8);
    table[tid] = xyzz_to_affine_c(r);
  }
};
#if !PS_GPU
template <class F> struct EmuParallel<FixedBaseTableK<F>> { static constexpr bool V = true; };   // host emulation only (backend.cuh)
#endif
// out[i] = scalar[i] * generator  (scalars: standard-form limbs), left in XYZZ form
template <class F>
struct FixedBaseMulK {
  static constexpr int BLOCK = 128;
  PS_DEV static void run(uint32_t i, const uint32_t* scalars, const Affine<F>* table, XYZZ<F>* out) {
    XYZZ<F> acc = XYZZ<F>::inf();
    for (int j = 0; j < 8; j++) {
      uint32_t limb = scalars[(size_t)i * 8 + j];
      for (int b = 0; b < 4; b++) {
        uint32_t d = (limb >> (8 * b)) & 0xFF;
        if (d) xyzz_madd_c(acc, table[(uint32_t)(4 * j + b) * 255 + d - 1]);
      }
    }
    out[i] = acc;
  }
};
// next[i] = 2^c * prev[i], left in XYZZ form
template <class F>
struct ShiftTableK {
  static constexpr int BLOCK = 128;
  PS_DEV static void run(uint32_t i, const Affine<F>* prev, XYZZ<F>* next, int c) {
    XYZZ<F> r = XYZZ<F>::from_affine(prev[i]);
    for (int d = 0; d < c; d++) r = xyzz_dbl_c(r);
    next[i] = r;
  }
};
// XYZZ -> affine for K consecutive points per thread with ONE field inversion (Montgomery's trick on ZZZ)
template <class F>
struct BatchToAffineK {
  static constexpr int BLOCK = 64;
  static constexpr uint32_t K = sizeof(F) == sizeof(Fp) ? 8 : 4;
  PS_DEV static void run(uint32_t t, uint32_t n, const XYZZ<F>* in, Affine<F>* out) {
    const uint32_t i0 = t * K;
    F pre[K];
    F acc = F::one();
#pragma unroll
    for (uint32_t k = 0; k < K; k++) {
      if (i0 + k < n) { F z = in[i0 + k].zzz; if (!in[i0 + k].zz.is_zero()) acc = acc * z; }
      pre[k] = acc;
    }
    F inv = FieldInv<F>::inv(acc);
#pragma unroll
    for (uint32_t kk = K; kk-- > 0;) {
      if (i0 + kk >= n) continue;
      XYZZ<F> p = in[i0 + kk];
      if (p.zz.is_zero()) { out[i0 + kk] = Affine<F>::inf(); continue; }
      F zzz_inv = kk > 0 ? inv * pre[kk - 1] : inv;
      inv = inv * p.zzz;
      F tt = zzz_inv * p.zz;
      out[i0 + kk] = Affine<F>{p.x * tt.sqr(), p.y * zzz_inv};
    }
  }
};

// Sums of the per-rank partial points of a sharded proof, read in place from the gathered records
// (stride bytes apart): item i adds, over all records, the points at byte offsets off0[i] and (if
// >= 0) off1[i].  One team of four lanes per item.
template <class F>
struct RecordSumK {
  static constexpr int BLOCK = 32;
  PS_DEV static void run(uint32_t tid, uint32_t count, const uint8_t* recs, uint32_t stride, int a0, int a1, int b0, int b1,
                         XYZZ<F>* out) {
    Coop<true> co(tid);
    if (co.idle()) return;
    const int o0 = tid == 0 ? a0 : b0, o1 = tid == 0 ? a1 : b1;
    XYZZ<F> r = XYZZ<F>::inf();
    for (uint32_t i = 0; i < count; i++) {
      const uint8_t* rec = recs + (size_t)i * stride;
      co.add(r, *(const XYZZ<F>*)(rec + o0));
      if (o1 >= 0) co.add(r, *(const XYZZ<F>*)(rec + o1));
    }
    if (co.writer()) out[tid] = r;
  }
};

// ---- GroupOps members ---------------------------------------------------------------------------------
template <class F>
int GroupOps<F>::msm_batch(ps_ctx* ctx, const MsmPlan& plan, const Affine<F>* slab, XYZZ<F>* d_out) {
  return msm_run_batch<F>(ctx, plan, slab, d_out);
}

template <class F>
int GroupOps<F>::decode(ps_ctx* ctx, const uint8_t* d_in, size_t n, int format, Affine<F>* d_out, uint32_t* d_err, bool subgroup_check,
                        uint8_t* d_status) {
  using DK = typename DecodeKernel<F>::K;
  PS_LAUNCH(DK, ctx->stream, n, d_in, format, d_out, d_err, subgroup_check ? 1 : 0, d_status);
  return PS_OK;
}

template <class F>
int GroupOps<F>::to_affine(ps_ctx* ctx, const XYZZ<F>* d_in, size_t n, Affine<F>* d_out) {
  PS_LAUNCH(BatchToAffineK<F>, ctx->stream, (n + BatchToAffineK<F>::K - 1) / BatchToAffineK<F>::K, (uint32_t)n, d_in, d_out);
  return PS_OK;
}

template <class F>
int GroupOps<F>::tables_finish(ps_ctx* ctx, Affine<F>* tab, size_t n, int c, int T) {
  if (T <= 1) return PS_OK;
  XYZZ<F>* tmp = ctx->arena.take<XYZZ<F>>(n);
  if (!tmp) return PS_ERR_ALLOC;
  const size_t groups = (n + BatchToAffineK<F>::K - 1) / BatchToAffineK<F>::K;
  for (int t = 1; t < T; t++) {
    PS_LAUNCH(ShiftTableK<F>, ctx->stream, n, (const Affine<F>*)(tab + (size_t)(t - 1) * n), tmp, c);
    PS_LAUNCH(BatchToAffineK<F>, ctx->stream, groups, (uint32_t)n, (const XYZZ<F>*)tmp, tab + (size_t)t * n);
  }
  return PS_OK;
}

template <class F>
int GroupOps<F>::from_scalars(ps_ctx* ctx, const uint32_t* d_scalars, size_t n, Affine<F>* d_out) {
  const int slot = PointBytes<F>::GROUP == PS_G1 ? 0 : 1;
  if (!ctx->fixed_base[slot]) {
    void* p = nullptr;
    PS_TRY(dev_alloc(&p, (size_t)32 * 255 * sizeof(Affine<F>)));
    ctx->fixed_base[slot] = p;
    PS_LAUNCH(FixedBaseTableK<F>, ctx->stream, (size_t)32 * 255, (Affine<F>*)p);
  }
  const Affine<F>* tbl = (const Affine<F>*)ctx->fixed_base[slot];
  XYZZ<F>* tmp = ctx->arena.take<XYZZ<F>>(n);
  if (!tmp) return PS_ERR_ALLOC;
  PS_LAUNCH(FixedBaseMulK<F>, ctx->stream, n, d_scalars, tbl, tmp);
  PS_LAUNCH(BatchToAffineK<F>, ctx->stream, (n + BatchToAffineK<F>::K - 1) / BatchToAffineK<F>::K, (uint32_t)n, (const XYZZ<F>*)tmp, d_out);
  return PS_OK;
}

template <class F>
int GroupOps<F>::encode_xyzz(ps_ctx* ctx, const XYZZ<F>* d_pts, size_t count, int format, uint8_t* d_bytes) {
  PS_LAUNCH(XyzzEncodeK<F>, ctx->stream, count, d_pts, format, d_bytes);
  return PS_OK;
}

template <class F>
int GroupOps<F>::encode_affine(ps_ctx* ctx, const Affine<F>* d_pts, size_t count, int format, uint8_t* d_bytes) {
  PS_LAUNCH(AffineEncodeK<F>, ctx->stream, count, d_pts, format, d_bytes);
  return PS_OK;
}

template <class F>
int GroupOps<F>::sum_points(ps_ctx* ctx, const XYZZ<F>* d_in, uint32_t count, XYZZ<F>* d_out) {
  return launch_coop<MsmSumK, F>(ctx->msm_team != 0, ctx->stream, 1, count, d_in, d_out);
}

template <class F>
int GroupOps<F>::record_sum(ps_ctx* ctx, int items, uint32_t count, const uint8_t* d_recs, uint32_t stride, const int off0[2],
                            const int off1[2], XYZZ<F>* d_out) {
  if (items < 1 || items > 2) return PS_ERR_ARG;
  PS_LAUNCH(RecordSumK<F>, ctx->stream, (size_t)items * TEAM, count, d_recs, stride, off0[0], off1[0], off0[items - 1], off1[items - 1], d_out);
  return PS_OK;
}

}  // namespace ps
