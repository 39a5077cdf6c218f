// What the orchestration code (capi.cu) needs from the Fr polynomial kernels: the QAP handle and the
// host-side entry points defined in capi_poly.cu, the translation unit that instantiates the NTT /
// interpolation / quotient kernels (ntt.cuh, poly.cuh, interp.cuh).
#pragma once
#include "context.cuh"

struct ps_qap {
  size_t n = 0, m = 0, n_io = 0;  // gates, variables, IO count
  int log_np = 0;                 // n' = 2^log_np >= n (transform size)
  bool dense = true;
  ps::Fr *left = nullptr, *right = nullptr, *out = nullptr;  // m x n, Montgomery (dense form)
  ps::NttTables tabs;
  ps::Fr* gpow = nullptr;       // g^k, k < n'
  ps::Fr* ginv_pow = nullptr;   // g^-k / n'
  ps::Fr* zinv_coset = nullptr; // 1 / z(g * omega^k), bit-reversed order
  ps::Fr* z_plain = nullptr;    // z(omega^k), bit-reversed order
  void* sparse = nullptr;       // ps::SparseQap* when built from a sparse R1CS (interp.cuh)
};

struct ps_bases {
  int group = 0;
  size_t n = 0;
  int c = 0;  // fixed window (0 = choose per call)
  int T = 1;  // precomputed tables
  void* tab = nullptr;    // T tables of n affine points
  void* slab = nullptr;   // the device allocation `tab` lives in: base sets of one slab can share an MSM pipeline
  bool owns = true;       // false: a view into a slab owned by a key
};

struct ps_g16_key {
  size_t n = 0, n_nio = 0;
  ps_bases *A = nullptr, *B = nullptr, *C = nullptr;
  void* slab_g1 = nullptr;   // A and C live in one allocation (their MSMs run as one batch)
};

struct ps_phgr13_key {
  size_t n = 0, n_mid = 0;
  ps_bases* g1[7] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};  // gsi vs ys vas was yas [vbs|wbs|ybs]
  ps_bases* ws = nullptr;
  void* slab_g1 = nullptr;   // the seven G1 base sets live in one allocation
};

namespace ps {

// witness -> device Montgomery; a, b, c, h on the device (n' entries each)
struct QuotientBufs { Fr *w, *a, *b, *c, *h; uint32_t* flag; uint32_t* enc_err; };
// quotient + the three MSM scalar vectors of the Groth16 proof (Montgomery form, arena memory)
struct G16Scalars { Fr *scA, *scB, *scC; size_t nA, nB, nC; QuotientBufs qb; };

// scalars (host, big-endian) -> device limbs; *d_err_out is set non-zero on the device for values >= r
int stage_scalars(ps_ctx* ctx, const uint8_t* scalars_be, size_t n, int mont, uint32_t** d_out, uint32_t** d_err_out);
int export_fr(ps_ctx* ctx, const Fr* d_src, size_t count, uint8_t* host_out);
int run_quotient(ps_ctx* ctx, const ps_qap* q, const uint8_t* witness_be, QuotientBufs* o, bool want_c = false);
int g16_build_scalars(ps_ctx* ctx, const ps_g16_key* key, const ps_qap* qap, const uint8_t* witness_be, const uint8_t* r_be,
                      const uint8_t* s_be, G16Scalars* o);

// Exponents of the trusted setups for a resident QAP (device memory, standard form; setup.cuh):
//   Groth16: pw[n] = x^k; pwt[n-1] = x^k t(x) / delta; lp[m] = (beta u_i + alpha v_i + w_i) / gamma (i < m - n_io) or / delta;
//            consts = alpha, beta, delta, gamma.       toxic = alpha, beta, delta, x, gamma (5 x 32 B big-endian)
struct G16SetupScalars { Fr *pw, *pwt, *lp, *consts; };
int g16_setup_scalars(ps_ctx* ctx, const ps_qap* q, const uint8_t* toxic_be, G16SetupScalars* o);
//   PHGR13: pw[n-1] = s^k; ek[k][m] for k = vs ws ys vas was yas vbs wbs ybs (every variable; the evaluation key uses the
//            last n_io); consts = av, aw, ay, gamma, beta*gamma, t(s)*ry.   toxic = s, av, aw, ay, rv, rw, beta, gamma
struct Phgr13SetupScalars { Fr* pw; Fr* ek[9]; Fr* consts; };
int phgr13_setup_scalars(ps_ctx* ctx, const ps_qap* q, const uint8_t* toxic_be, Phgr13SetupScalars* o);

// (capi.cu) `rows` MSMs over all points of one base set of group F (Fp: G1, Fp2: G2), row k's scalars at
// d_scalars + k * b->n * 8 (limbs), result k to d_out[k]; all rows run as one pipeline (MsmPlan's row mode), split into
// several only where one pipeline's entry or bucket count would reach 2^31
template <class F> struct XYZZ;
template <class F> int msm_rows(ps_ctx* ctx, const ps_bases* b, const uint32_t* d_scalars, size_t rows, int mont, XYZZ<F>* d_out);
// (capi.cu) window of a batch of `nsets` MSMs over `total_points` points in all, for base sets with all window tables
int batch_window(ps_ctx* ctx, size_t total_points, int nsets);

// host-only helpers shared by both translation units
inline int parse_fr(const uint8_t* src, Fr* out) {   // 32 B big-endian, canonical -> Montgomery
  Fr x;
  for (int j = 0; j < 8; j++) {
    const uint8_t* p = src + 4 * (7 - j);
    x.v[j] = ((uint32_t)p[0] << 24) | ((uint32_t)p[1] << 16) | ((uint32_t)p[2] << 8) | (uint32_t)p[3];
  }
  bool lt = false;
  for (int j = 7; j >= 0; j--) {
    const uint32_t m = FrParams::MOD(j);
    if (x.v[j] != m) { lt = x.v[j] < m; break; }
  }
  if (!lt) return PS_ERR_ENCODING;
  *out = x.to_mont();
  return PS_OK;
}
inline int check_err_flag(ps_ctx* ctx, const uint32_t* d_err, int code) {
  uint32_t h = 0;
  PS_TRY(dev_d2h(&h, d_err, 4, ctx->stream));
  PS_TRY(dev_sync(ctx->stream));
  return h ? code : PS_OK;
}
inline int begin_call(ps_ctx* ctx) {
  if (!ctx) return PS_ERR_ARG;
#if PS_GPU
  PS_CUDA_TRY(cudaSetDevice(ctx->device));
#endif
  PS_TRY(ctx->arena2.reset());
  return ctx->arena.reset();
}
inline int log2_exact(size_t v) {
  int l = 0;
  while (((size_t)1 << l) < v) l++;
  return ((size_t)1 << l) == v ? l : -1;
}

}  // namespace ps
