// C ABI, part 4: the verifiers (SURVEY 8 f4) -- pairing-product checks on the device and, on top of them and of
// the MSM entry points, Groth16Verify (groth16.go:214-233) and PHGR13Verify (pinochio.go:281-375).
//
// Every equation the reference tests, "left.Equal(right)" over GT values, is rewritten as  prod_i e(P_i, Q_i) == 1
// with the G1 points of one side negated; the sums over the public inputs (sum_i io_i IoLP_i, computeCommitIOSolution
// pinochio.go:390-407) and the point additions around them are MSMs with the extra points given the scalar 1.
// One thread per Miller loop, one per final exponentiation (pairing.cuh): the work per proof is constant, the
// parallelism is across pairs, equations and the proofs of a batch.
#include "group_ops.cuh"
#include "pairing.cuh"
#include "poly_api.cuh"
#include "verify_batch.cuh"
#include "verify_batch_phgr13.cuh"

#include <errno.h>
#include <sys/random.h>
#include <vector>

using namespace ps;

namespace {

inline size_t g1_bytes(int format) { return format == PS_FMT_COMPRESSED ? 48 : 96; }
inline size_t g2_bytes(int format) { return format == PS_FMT_COMPRESSED ? 96 : 192; }

// -P for a point in wire format: the sign flag of the compressed form (bit 5 of byte 0; infinity has none),
// p - y for the uncompressed one (big-endian subtraction; y = 0 cannot occur on these curves)
void negate_point(uint8_t* pt, int group, int format) {
  if (pt[0] & 0x40) return;                       // infinity
  if (format == PS_FMT_COMPRESSED) { pt[0] ^= 0x20; return; }
  static const uint8_t P_BE[48] = {0x1a, 0x01, 0x11, 0xea, 0x39, 0x7f, 0xe6, 0x9a, 0x4b, 0x1b, 0xa7, 0xb6, 0x43, 0x4b, 0xac, 0xd7,
                                   0x64, 0x77, 0x4b, 0x84, 0xf3, 0x85, 0x12, 0xbf, 0x67, 0x30, 0xd2, 0xa0, 0xf6, 0xb0, 0xf6, 0x24,
                                   0x1e, 0xab, 0xff, 0xfe, 0xb1, 0x53, 0xff, 0xff, 0xb9, 0xfe, 0xff, 0xff, 0xff, 0xff, 0xaa, 0xab};
  const int coords = group == PS_G1 ? 1 : 2;      // y is the second half: 48 B (G1) or 2 x 48 B (G2: c1 | c0)
  uint8_t* y = pt + 48 * coords;
  for (int c = 0; c < coords; c++, y += 48) {
    bool zero = true;
    for (int i = 0; i < 48; i++) zero = zero && y[i] == 0;
    if (zero) continue;
    int borrow = 0;
    for (int i = 47; i >= 0; i--) {
      int d = (int)P_BE[i] - (int)y[i] - borrow;
      borrow = d < 0;
      y[i] = (uint8_t)(d + (borrow ? 256 : 0));
    }
  }
}

// sum_i scalars[i] * points[i] through the public MSM path; result as wire bytes of the same format's COMPRESSED size
// (ps_msm returns compressed points)
int msm_bytes(ps_ctx* ctx, int group, const std::vector<uint8_t>& points, const std::vector<uint8_t>& scalars_be, size_t n, int format,
              uint8_t* out) {
  ps_bases* b = nullptr;
  PS_TRY(ps_bases_load(ctx, group, points.data(), n, format, 0, 1, &b));
  int rc = ps_msm(ctx, b, scalars_be.data(), n, out);
  ps_bases_free(b);
  return rc;
}

const uint8_t ONE_BE[32] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 1};

// the generator of G2 in compressed wire format (NewG2().Base(), curve.go:30)
int g2_generator_bytes(ps_ctx* ctx, uint8_t out[96]) {
  ps_bases* b = nullptr;
  PS_TRY(ps_bases_from_scalars(ctx, PS_G2, ONE_BE, 1, 0, 1, &b));
  int rc = ps_bases_export(ctx, b, 0, 1, PS_FMT_COMPRESSED, out);
  ps_bases_free(b);
  return rc;
}

// largest batch of ps_g16_verify_batch: the per-proof device state of 2^20 proofs (tree nodes, points, Miller values) is about 3 GB
constexpr size_t VERIFY_BATCH_MAX = size_t(1) << 20;

// n nonzero 128-bit weights from the operating system's generator, as 4 little-endian limbs each
int draw_weights(size_t n, std::vector<uint32_t>& limbs) {
  for (size_t i = 0; i < n; i++) {
    uint32_t* k = limbs.data() + 4 * i;
    do {
      size_t got = 0;
      while (got < 16) {
        ssize_t r = getrandom((uint8_t*)k + got, 16 - got, 0);
        if (r < 0 && errno == EINTR) continue;
        if (r <= 0) return PS_ERR_UNSUPPORTED;
        got += (size_t)r;
      }
    } while ((k[0] | k[1] | k[2] | k[3]) == 0);
  }
  return PS_OK;
}

// Device state of one ps_g16_verify_batch call (arena memory); check_nodes runs the node check of the listed nodes
struct VbState {
  ps_ctx* ctx;
  const ps_bases* iolp;    // null when n_io == 0
  uint32_t n, P, n_io;
  const Fr* io;            // n x n_io, Montgomery
  const Fr* w;             // per-proof weights (0 for a proof that did not decode)
  Fp12* f; G1XYZZ* cs; Fr* s;
  Fp12* fe; uint8_t* bad;  // per node: value after the final exponentiation, check failed
  const G1Affine* alpha; const G2Affine* key2;

  int check_nodes(const std::vector<uint32_t>& nodes) {
    const size_t m = nodes.size();
    Arena& ar = ctx->arena;
    ps_stream_t st = ctx->stream;
    uint32_t* d_nodes = ar.take<uint32_t>(m);
    G1XYZZ* L = ar.take<G1XYZZ>(m);
    G1XYZZ* p = ar.take<G1XYZZ>(3 * m);
    G1Affine* pa = ar.take<G1Affine>(3 * m);
    G2Affine* q = ar.take<G2Affine>(3 * m);
    Fp12* fm = ar.take<Fp12>(3 * m);
    Fp12* acc = ar.take<Fp12>(m);
    Fr* sc = n_io ? ar.take<Fr>(m * n_io) : nullptr;
    if (!d_nodes || !L || !p || !pa || !q || !fm || !acc || (n_io && !sc)) return PS_ERR_ALLOC;
    PS_TRY(dev_h2d(d_nodes, nodes.data(), m * 4, st));
    if (n_io) {
      PS_LAUNCH(VbIoCombineK, st, m * n_io, n_io, P, n, (const uint32_t*)d_nodes, io, w, sc);
      PS_TRY(msm_rows<Fp>(ctx, iolp, (const uint32_t*)sc, m, 0, L));
    } else {
      PS_TRY(dev_memset(L, 0, m * sizeof(G1XYZZ), st));
    }
    PS_LAUNCH(VbNodePointsK, st, m, (const uint32_t*)d_nodes, (const Fr*)s, (const G1XYZZ*)cs, (const G1XYZZ*)L, alpha, key2, p, q);
    PS_TRY(GroupOps<Fp>::to_affine(ctx, p, 3 * m, pa));
    PS_LAUNCH(PairingMillerK, st, 3 * m, (const G1Affine*)pa, (const G2Affine*)q, fm);
    PS_LAUNCH(VbNodeProductK, st, m, (const uint32_t*)d_nodes, (const Fp12*)f, (const Fp12*)fm, acc);
    PS_LAUNCH(VbFinalExpK, st, m, (const Fp12*)acc, fm);                   // the Miller values are consumed: reuse fm[0, m)
    PS_LAUNCH(VbVerdictK, st, m, (const uint32_t*)d_nodes, (const Fp12*)fm, fe, bad);
    return PS_OK;
  }
};

// Device state of one ps_phgr13_verify_batch call (arena memory); check_nodes runs the node check of the listed nodes
struct PvState {
  ps_ctx* ctx;
  const ps_bases* ys;      // null when n_io == 0
  uint32_t n, P, n_io;
  const Fr* io;            // n x n_io, Montgomery
  const Fr* w1;            // per-proof rho_i1 (0 for a proof that did not decode)
  Fp12* f; G1XYZZ* s1; G2XYZZ* s2;
  Fp12* fe; uint8_t* bad;  // per node: value after the final exponentiation, check failed
  const G1Affine* key1; const G2Affine* key2;

  int check_nodes(const std::vector<uint32_t>& nodes) {
    const size_t m = nodes.size();
    Arena& ar = ctx->arena;
    ps_stream_t st = ctx->stream;
    uint32_t* d_nodes = ar.take<uint32_t>(m);
    G1XYZZ* L = ar.take<G1XYZZ>(m);
    G1XYZZ* p = ar.take<G1XYZZ>(8 * m);
    G2XYZZ* q = ar.take<G2XYZZ>(8 * m);
    G1Affine* pa = ar.take<G1Affine>(8 * m);
    G2Affine* qa = ar.take<G2Affine>(8 * m);
    Fp12* fm = ar.take<Fp12>(8 * m);
    Fp12* acc = ar.take<Fp12>(m);
    Fr* sc = n_io ? ar.take<Fr>(m * n_io) : nullptr;
    if (!d_nodes || !L || !p || !q || !pa || !qa || !fm || !acc || (n_io && !sc)) return PS_ERR_ALLOC;
    PS_TRY(dev_h2d(d_nodes, nodes.data(), m * 4, st));
    if (n_io) {
      PS_LAUNCH(VbIoCombineK, st, m * n_io, n_io, P, n, (const uint32_t*)d_nodes, io, w1, sc);
      PS_TRY(msm_rows<Fp>(ctx, ys, (const uint32_t*)sc, m, 0, L));
    } else {
      PS_TRY(dev_memset(L, 0, m * sizeof(G1XYZZ), st));
    }
    PS_LAUNCH(PvNodePointsK, st, m, P, (const uint32_t*)d_nodes, (const G1XYZZ*)s1, (const G2XYZZ*)s2, (const G1XYZZ*)L, key1, key2, p, q);
    PS_TRY(GroupOps<Fp>::to_affine(ctx, p, 8 * m, pa));
    PS_TRY(GroupOps<Fp2>::to_affine(ctx, q, 8 * m, qa));
    PS_LAUNCH(PairingMillerK, st, 8 * m, (const G1Affine*)pa, (const G2Affine*)qa, fm);
    PS_LAUNCH(PvNodeProductK, st, m, (const uint32_t*)d_nodes, (const Fp12*)f, (const Fp12*)fm, acc);
    PS_LAUNCH(VbFinalExpK, st, m, (const Fp12*)acc, fm);                   // the Miller values are consumed: reuse fm[0, m)
    PS_LAUNCH(VbVerdictK, st, m, (const uint32_t*)d_nodes, (const Fp12*)fm, fe, bad);
    return PS_OK;
  }
};

// Per-proof verdicts after a failed root check: level by level, only below failing nodes; one node check per failing
// node (its left child), the right child's value follows as parent * conj(left).  Proofs under a failing leaf get 0.
template <class State>
int bisect(State& vs, ps_ctx* ctx, uint32_t P, uint32_t n, const uint8_t* d_bad, bool root_bad, uint8_t* per_proof) {
  std::vector<uint32_t> failing;
  if (root_bad) failing.push_back(1);
  std::vector<uint8_t> hbad;
  while (!failing.empty() && failing[0] < P) {
    std::vector<uint32_t> lefts(failing.size());
    for (size_t t = 0; t < failing.size(); t++) lefts[t] = 2 * failing[t];
    PS_TRY(vs.check_nodes(lefts));
    uint32_t level_first = 1;
    while (level_first * 2 <= lefts[0]) level_first <<= 1;   // first node of the children's level
    hbad.resize(level_first);
    PS_TRY(dev_d2h(hbad.data(), d_bad + level_first, level_first, ctx->stream));
    PS_TRY(dev_sync(ctx->stream));
    std::vector<uint32_t> next;
    for (uint32_t k : lefts)
      for (uint32_t c = k; c <= k + 1; c++)
        if (hbad[c - level_first]) next.push_back(c);
    failing.swap(next);
  }
  for (uint32_t k : failing)
    if (k >= P && k - P < n) per_proof[k - P] = 0;
  return PS_OK;
}

// big-endian 16-byte weights -> 4 little-endian limbs each; PS_ERR_ARG on a zero weight
int parse_weights(const uint8_t* weights, size_t count, std::vector<uint32_t>& limbs) {
  for (size_t i = 0; i < count; i++) {
    const uint8_t* b = weights + 16 * i;
    uint32_t* k = limbs.data() + 4 * i;
    for (int j = 0; j < 4; j++)
      k[j] = ((uint32_t)b[12 - 4 * j] << 24) | ((uint32_t)b[13 - 4 * j] << 16) | ((uint32_t)b[14 - 4 * j] << 8) | b[15 - 4 * j];
    if ((k[0] | k[1] | k[2] | k[3]) == 0) return PS_ERR_ARG;
  }
  return PS_OK;
}

}  // namespace

extern "C" {

int ps_pairing_check_batch(ps_ctx* ctx, const uint8_t* g1_points, const uint8_t* g2_points, const uint32_t* counts, size_t n_checks,
                           int format, uint8_t* ok) {
  if (!ctx || !counts || !ok || (format != PS_FMT_COMPRESSED && format != PS_FMT_AFFINE)) return PS_ERR_ARG;
  if (n_checks == 0) return PS_OK;
  if (n_checks > (1u << 24)) return PS_ERR_UNSUPPORTED;
  std::vector<uint32_t> first(n_checks + 1, 0);
  for (size_t t = 0; t < n_checks; t++) {
    if (counts[t] > (1u << 20)) return PS_ERR_UNSUPPORTED;
    first[t + 1] = first[t] + counts[t];
    if (first[t + 1] > (1u << 26)) return PS_ERR_UNSUPPORTED;
  }
  const size_t total = first[n_checks];
  if (total && (!g1_points || !g2_points)) return PS_ERR_ARG;
  PS_TRY(begin_call(ctx));
  ps_stream_t st = ctx->stream;
  Arena& ar = ctx->arena;
  const size_t b1 = total * g1_bytes(format), b2 = total * g2_bytes(format);
  uint8_t* d_in1 = ar.take<uint8_t>(b1);
  uint8_t* d_in2 = ar.take<uint8_t>(b2);
  G1Affine* P = ar.take<G1Affine>(total);
  G2Affine* Q = ar.take<G2Affine>(total);
  Fp12* f = ar.take<Fp12>(total);
  uint32_t* d_first = ar.take<uint32_t>(n_checks + 1);
  uint8_t* d_ok = ar.take<uint8_t>(n_checks);
  uint32_t* d_err = ar.take<uint32_t>(1);
  if (!d_in1 || !d_in2 || !P || !Q || !f || !d_first || !d_ok || !d_err) return PS_ERR_ALLOC;
  PS_TRY(dev_memset(d_err, 0, 4, st));
  if (total) {
    PS_TRY(dev_h2d(d_in1, g1_points, b1, st));
    PS_TRY(dev_h2d(d_in2, g2_points, b2, st));
    PS_TRY(GroupOps<Fp>::decode(ctx, d_in1, total, format, P, d_err, ctx->subgroup_check != 0));
    PS_TRY(GroupOps<Fp2>::decode(ctx, d_in2, total, format, Q, d_err, ctx->subgroup_check != 0));
  }
  PS_TRY(dev_h2d(d_first, first.data(), (n_checks + 1) * 4, st));
  PS_LAUNCH(PairingMillerK, st, total, (const G1Affine*)P, (const G2Affine*)Q, f);
  PS_LAUNCH(PairingCheckK, st, n_checks, (const Fp12*)f, (const uint32_t*)d_first, d_ok);
  PS_TRY(dev_d2h(ok, d_ok, n_checks, st));
  return check_err_flag(ctx, d_err, PS_ERR_ENCODING);   // synchronises: `first` and `ok` are settled
}

int ps_g16_verify(ps_ctx* ctx, const uint8_t* alpha, const uint8_t* beta2, const uint8_t* gamma2, const uint8_t* delta2,
                  const uint8_t* iolp, size_t n_io, const uint8_t* io_be, const uint8_t* A, const uint8_t* B, const uint8_t* C, int* ok) {
  if (!ctx || !alpha || !beta2 || !gamma2 || !delta2 || !A || !B || !C || !ok || (n_io && (!iolp || !io_be))) return PS_ERR_ARG;
  *ok = 0;
  // b1 = sum_i io[i] * IoLP[i]   (groth16.go:224-227)
  uint8_t b1[48];
  if (n_io) {
    std::vector<uint8_t> pts(iolp, iolp + n_io * 48), sc(io_be, io_be + n_io * 32);
    PS_TRY(msm_bytes(ctx, PS_G1, pts, sc, n_io, PS_FMT_COMPRESSED, b1));
  } else {
    memset(b1, 0, 48);
    b1[0] = 0xc0;
  }
  // e(A, B) == e(Alpha, Beta2) e(b1, Gamma) e(C, Delta2)   <=>   e(-A, B) e(Alpha, Beta2) e(b1, Gamma) e(C, Delta2) == 1
  uint8_t g1[4 * 48], g2[4 * 96];
  memcpy(g1, A, 48); negate_point(g1, PS_G1, PS_FMT_COMPRESSED);
  memcpy(g1 + 48, alpha, 48); memcpy(g1 + 96, b1, 48); memcpy(g1 + 144, C, 48);
  memcpy(g2, B, 96); memcpy(g2 + 96, beta2, 96); memcpy(g2 + 192, gamma2, 96); memcpy(g2 + 288, delta2, 96);
  const uint32_t count = 4;
  uint8_t res = 0;
  PS_TRY(ps_pairing_check_batch(ctx, g1, g2, &count, 1, PS_FMT_COMPRESSED, &res));
  *ok = res ? 1 : 0;
  return PS_OK;
}

int ps_g16_verify_batch(ps_ctx* ctx, const uint8_t* alpha, const uint8_t* beta2, const uint8_t* gamma2, const uint8_t* delta2,
                        const uint8_t* iolp, size_t n_io, size_t n_proofs, const uint8_t* io_be, const uint8_t* A, const uint8_t* B,
                        const uint8_t* C, const uint8_t* weights, int* ok, uint8_t* per_proof) {
  if (!ctx || !alpha || !beta2 || !gamma2 || !delta2 || !ok || (n_io && !iolp)) return PS_ERR_ARG;
  if (n_proofs && (!A || !B || !C || (n_io && !io_be))) return PS_ERR_ARG;
  *ok = 0;
  if (n_proofs > VERIFY_BATCH_MAX || n_io > (1u << 26) || (unsigned long long)n_proofs * n_io >= (1ull << 31))
    return PS_ERR_UNSUPPORTED;
  std::vector<uint32_t> rho(4 * n_proofs);
  if (weights) PS_TRY(parse_weights(weights, n_proofs, rho));
  if (n_proofs == 0) { *ok = 1; return PS_OK; }
  if (!weights) PS_TRY(draw_weights(n_proofs, rho));
  // the key's IoLP as a base set: decoding errors of key points are the caller's (PS_ERR_ENCODING)
  ps_bases* bl = nullptr;
  if (n_io) PS_TRY(ps_bases_load(ctx, PS_G1, iolp, n_io, PS_FMT_COMPRESSED, 0, 1, &bl));
  struct Free { ps_bases* b; ~Free() { ps_bases_free(b); } } free_bl{bl};
  PS_TRY(begin_call(ctx));
  ctx->evv_valid = false;
  ps_stream_t st = ctx->stream;
  Arena& ar = ctx->arena;
  const uint32_t n = (uint32_t)n_proofs;
  uint32_t P = 1;
  while (P < n) P <<= 1;
  uint8_t* d_key = ar.take<uint8_t>(48 + 3 * 96);
  uint8_t* d_pts = ar.take<uint8_t>(n_proofs * (48 + 96 + 48));
  uint32_t* d_rho = ar.take<uint32_t>(4 * n_proofs);
  G1Affine* d_alpha = ar.take<G1Affine>(1);
  G2Affine* d_key2 = ar.take<G2Affine>(3);
  G1Affine* d_A = ar.take<G1Affine>(n);
  G1Affine* d_C = ar.take<G1Affine>(n);
  G2Affine* d_B = ar.take<G2Affine>(P);
  uint8_t* d_st = ar.take<uint8_t>(3 * n_proofs);
  Fr* d_w = ar.take<Fr>(n);
  uint8_t* d_valid = ar.take<uint8_t>(n);
  G1XYZZ* d_negA = ar.take<G1XYZZ>(P);
  G1Affine* d_negAa = ar.take<G1Affine>(P);
  Fp12* d_f = ar.take<Fp12>(2 * P);
  G1XYZZ* d_cs = ar.take<G1XYZZ>(2 * P);
  Fr* d_s = ar.take<Fr>(2 * P);
  Fp12* d_fe = ar.take<Fp12>(2 * P);
  uint8_t* d_bad = ar.take<uint8_t>(2 * P);
  uint32_t* d_err = ar.take<uint32_t>(1);   // key points; proof points report per proof
  if (!d_key || !d_pts || !d_rho || !d_alpha || !d_key2 || !d_A || !d_C || !d_B || !d_st || !d_w ||
      !d_valid || !d_negA || !d_negAa || !d_f || !d_cs || !d_s || !d_fe || !d_bad || !d_err)
    return PS_ERR_ALLOC;
  PS_TRY(ctx_verify_event(ctx, 0));
  std::vector<uint8_t> key(48 + 3 * 96);
  memcpy(key.data(), alpha, 48); memcpy(key.data() + 48, beta2, 96); memcpy(key.data() + 144, gamma2, 96);
  memcpy(key.data() + 240, delta2, 96);
  PS_TRY(dev_h2d(d_key, key.data(), key.size(), st));
  PS_TRY(dev_h2d(d_pts, A, n_proofs * 48, st));
  PS_TRY(dev_h2d(d_pts + n_proofs * 48, C, n_proofs * 48, st));
  PS_TRY(dev_h2d(d_pts + n_proofs * 96, B, n_proofs * 96, st));
  PS_TRY(dev_h2d(d_rho, rho.data(), rho.size() * 4, st));
  PS_TRY(dev_memset(d_err, 0, 4, st));
  PS_TRY(dev_memset(d_bad, 0, 2 * P, st));
  if (P > n) PS_TRY(dev_memset(d_B + n, 0, (P - n) * sizeof(G2Affine), st));   // empty slots pair with infinity
  PS_TRY(ctx_verify_event(ctx, 1));
  // key points follow the context's subgroup_check; proof points are untrusted and always checked, with a status each
  const bool sub = ctx->subgroup_check != 0;
  PS_TRY(GroupOps<Fp>::decode(ctx, d_key, 1, PS_FMT_COMPRESSED, d_alpha, d_err, sub));
  PS_TRY(GroupOps<Fp2>::decode(ctx, d_key + 48, 3, PS_FMT_COMPRESSED, d_key2, d_err, sub));
  uint32_t* d_perr = ar.take<uint32_t>(1);
  if (!d_perr) return PS_ERR_ALLOC;
  PS_TRY(GroupOps<Fp>::decode(ctx, d_pts, n, PS_FMT_COMPRESSED, d_A, d_perr, true, d_st));
  PS_TRY(GroupOps<Fp2>::decode(ctx, d_pts + n_proofs * 96, n, PS_FMT_COMPRESSED, d_B, d_perr, true, d_st + n_proofs));
  PS_TRY(GroupOps<Fp>::decode(ctx, d_pts + n_proofs * 48, n, PS_FMT_COMPRESSED, d_C, d_perr, true, d_st + 2 * n_proofs));
  PS_TRY(ctx_verify_event(ctx, 2));
  PS_LAUNCH(VbWeighK, st, P, n, P, (const uint32_t*)d_rho, (const uint8_t*)d_st, (const G1Affine*)d_A, (const G1Affine*)d_C, d_negA, d_cs,
            d_s, d_w, d_valid);
  PS_TRY(GroupOps<Fp>::to_affine(ctx, d_negA, P, d_negAa));
  PS_TRY(ctx_verify_event(ctx, 3));
  uint32_t *d_io = nullptr, *d_ioerr = nullptr;
  if (n_io) PS_TRY(stage_scalars(ctx, io_be, n_proofs * n_io, 1, &d_io, &d_ioerr));
  VbState vs{ctx, bl, n, P, (uint32_t)n_io, (const Fr*)d_io, d_w, d_f, d_cs, d_s, d_fe, d_bad, d_alpha, d_key2};
  PS_TRY(ctx_verify_event(ctx, 4));   // the io sums of the root run inside its node check (phase 6)
  PS_LAUNCH(PairingMillerK, st, P, (const G1Affine*)d_negAa, (const G2Affine*)d_B, d_f + P);
  PS_TRY(ctx_verify_event(ctx, 5));
  for (uint32_t first = P >> 1; first >= 1; first >>= 1) PS_LAUNCH(VbTreeLevelK, st, first, first, d_f, d_cs, d_s);
  PS_TRY(ctx_verify_event(ctx, 6));
  PS_TRY(vs.check_nodes(std::vector<uint32_t>{1}));
  PS_TRY(ctx_verify_event(ctx, 7));
  std::vector<uint8_t> valid(n_proofs);
  uint8_t root_bad = 0;
  PS_TRY(dev_d2h(valid.data(), d_valid, n_proofs, st));
  PS_TRY(dev_d2h(&root_bad, d_bad + 1, 1, st));
  uint32_t herr[2] = {0, 0};
  PS_TRY(dev_d2h(herr, d_err, 4, st));
  if (n_io) PS_TRY(dev_d2h(herr + 1, d_ioerr, 4, st));
  PS_TRY(dev_sync(st));
  if (herr[0] || herr[1]) return PS_ERR_ENCODING;
  bool all_valid = true;
  for (size_t i = 0; i < n_proofs; i++) all_valid = all_valid && valid[i];
  *ok = (all_valid && !root_bad) ? 1 : 0;
  if (per_proof) {
    memcpy(per_proof, valid.data(), n_proofs);
    PS_TRY(bisect(vs, ctx, P, n, d_bad, root_bad != 0, per_proof));
  }
  PS_TRY(ctx_verify_event(ctx, 8));
  ctx->evv_valid = true;
  return PS_OK;
}

int ps_phgr13_verify(ps_ctx* ctx, const uint8_t* vk_fixed, const uint8_t* vs, const uint8_t* ws, const uint8_t* ys, size_t n_io,
                     const uint8_t* io_be, const uint8_t* proof, int* ok) {
  if (!ctx || !vk_fixed || !proof || !ok || (n_io && (!vs || !ws || !ys || !io_be))) return PS_ERR_ARG;
  *ok = 0;
  // vk_fixed: av(G2) aw(G1) ay(G2) gamma(G2) bgamma(G1) bgamma2(G2) yts(G2)     (layout of ps_phgr13_setup)
  const uint8_t *av = vk_fixed, *aw = vk_fixed + 96, *ay = vk_fixed + 144, *gamma = vk_fixed + 240, *bgamma = vk_fixed + 336,
                *bgamma2 = vk_fixed + 384, *yts = vk_fixed + 480;
  // proof: the 432 bytes ps_phgr13_prove writes -- hs vss yss vass wass yass gz (G1) then wss (G2)
  const uint8_t *hs = proof, *vss = proof + 48, *yss = proof + 96, *vass = proof + 144, *wass = proof + 192, *yass = proof + 240,
                *gz = proof + 288, *wss = proof + 336;
  // gv = sum io_k vs_k + vss, gw = sum io_k ws_k + wss, gy = sum io_k ys_k + yss      (pinochio.go:293-308)
  std::vector<uint8_t> sc(io_be, io_be + n_io * 32);
  sc.insert(sc.end(), ONE_BE, ONE_BE + 32);
  uint8_t gv[48], gw[96], gy[48], lt1[48], g2gen[96];
  {
    std::vector<uint8_t> pts(vs, vs + n_io * 48);
    pts.insert(pts.end(), vss, vss + 48);
    PS_TRY(msm_bytes(ctx, PS_G1, pts, sc, n_io + 1, PS_FMT_COMPRESSED, gv));
  }
  {
    std::vector<uint8_t> pts(ws, ws + n_io * 96);
    pts.insert(pts.end(), wss, wss + 96);
    PS_TRY(msm_bytes(ctx, PS_G2, pts, sc, n_io + 1, PS_FMT_COMPRESSED, gw));
  }
  {
    std::vector<uint8_t> pts(ys, ys + n_io * 48);
    pts.insert(pts.end(), yss, yss + 48);
    PS_TRY(msm_bytes(ctx, PS_G1, pts, sc, n_io + 1, PS_FMT_COMPRESSED, gy));
  }
  {   // lt1 = vss + yss   (pinochio.go:365)
    std::vector<uint8_t> pts(vss, vss + 48), one2(ONE_BE, ONE_BE + 32);
    pts.insert(pts.end(), yss, yss + 48);
    one2.insert(one2.end(), ONE_BE, ONE_BE + 32);
    PS_TRY(msm_bytes(ctx, PS_G1, pts, one2, 2, PS_FMT_COMPRESSED, lt1));
  }
  PS_TRY(g2_generator_bytes(ctx, g2gen));
  // the five equations of pinochio.go:312-372, each as a product that must be 1
  std::vector<uint8_t> g1, g2;
  auto pair = [&](const uint8_t* p, bool neg, const uint8_t* q) {
    uint8_t t[48];
    memcpy(t, p, 48);
    if (neg) negate_point(t, PS_G1, PS_FMT_COMPRESSED);
    g1.insert(g1.end(), t, t + 48);
    g2.insert(g2.end(), q, q + 96);
  };
  pair(gv, false, gw); pair(hs, true, yts); pair(gy, true, g2gen);            // division check
  pair(vass, false, g2gen); pair(vss, true, av);                                // CRS checks
  pair(wass, false, g2gen); pair(aw, true, wss);
  pair(yass, false, g2gen); pair(yss, true, ay);
  pair(gz, false, gamma); pair(lt1, true, bgamma2); pair(bgamma, true, wss);    // linear check
  const uint32_t counts[5] = {3, 2, 2, 2, 3};
  uint8_t res[5] = {0, 0, 0, 0, 0};
  PS_TRY(ps_pairing_check_batch(ctx, g1.data(), g2.data(), counts, 5, PS_FMT_COMPRESSED, res));
  *ok = (res[0] && res[1] && res[2] && res[3] && res[4]) ? 1 : 0;
  return PS_OK;
}

int ps_phgr13_verify_batch(ps_ctx* ctx, const uint8_t* vk_fixed, const uint8_t* vs, const uint8_t* ws, const uint8_t* ys, size_t n_io,
                           size_t n_proofs, const uint8_t* io_be, const uint8_t* proofs, const uint8_t* weights, int* ok,
                           uint8_t* per_proof) {
  if (!ctx || !vk_fixed || !ok || (n_io && (!vs || !ws || !ys))) return PS_ERR_ARG;
  if (n_proofs && (!proofs || (n_io && !io_be))) return PS_ERR_ARG;
  *ok = 0;
  if (n_proofs > VERIFY_BATCH_MAX || n_io > (1u << 26) || (unsigned long long)n_proofs * n_io >= (1ull << 31))
    return PS_ERR_UNSUPPORTED;
  std::vector<uint32_t> rho(20 * n_proofs);
  if (weights) PS_TRY(parse_weights(weights, 5 * n_proofs, rho));
  if (n_proofs == 0) { *ok = 1; return PS_OK; }
  if (!weights) PS_TRY(draw_weights(5 * n_proofs, rho));
  // key material first (these calls reset the scratch arena): G2gen, and vs / ws / ys as base sets with all window
  // tables, the window chosen for n_proofs io rows (decoding errors of key points are the caller's: PS_ERR_ENCODING)
  uint8_t g2gen[96];
  PS_TRY(g2_generator_bytes(ctx, g2gen));
  ps_bases *bv = nullptr, *bw = nullptr, *by = nullptr;
  struct Free { ps_bases** b[3]; ~Free() { for (auto p : b) ps_bases_free(*p); } } free_b{{&bv, &bw, &by}};
  if (n_io) {
    const int c = batch_window(ctx, n_proofs * n_io, (int)n_proofs);
    PS_TRY(ps_bases_load(ctx, PS_G1, vs, n_io, PS_FMT_COMPRESSED, c, -1, &bv));
    PS_TRY(ps_bases_load(ctx, PS_G2, ws, n_io, PS_FMT_COMPRESSED, c, -1, &bw));
    PS_TRY(ps_bases_load(ctx, PS_G1, ys, n_io, PS_FMT_COMPRESSED, c, -1, &by));
  }
  PS_TRY(begin_call(ctx));
  ctx->evv_valid = false;
  ps_stream_t st = ctx->stream;
  Arena& ar = ctx->arena;
  const uint32_t n = (uint32_t)n_proofs;
  uint32_t P = 1;
  while (P < n) P <<= 1;
  // vk_fixed: av(G2) aw(G1) ay(G2) gamma(G2) bgamma(G1) bgamma2(G2) yts(G2); on the device key1 = aw bgamma,
  // key2 = av ay gamma bgamma2 yts G2gen
  std::vector<uint8_t> key(2 * 48 + 6 * 96);
  memcpy(key.data(), vk_fixed + 96, 48); memcpy(key.data() + 48, vk_fixed + 336, 48);
  const size_t g2_off[5] = {0, 144, 240, 384, 480};
  for (int j = 0; j < 5; j++) memcpy(key.data() + 96 + 96 * j, vk_fixed + g2_off[j], 96);
  memcpy(key.data() + 96 + 5 * 96, g2gen, 96);
  // proof points regrouped by field: the seven G1 fields (hs vss yss vass wass yass gz) field-major, then wss
  std::vector<uint8_t> pts(n_proofs * 432);
  for (size_t i = 0; i < n_proofs; i++) {
    for (int j = 0; j < 7; j++) memcpy(pts.data() + (j * n_proofs + i) * 48, proofs + 432 * i + 48 * j, 48);
    memcpy(pts.data() + 7 * 48 * n_proofs + 96 * i, proofs + 432 * i + 336, 96);
  }
  uint8_t* d_key = ar.take<uint8_t>(key.size());
  uint8_t* d_pts = ar.take<uint8_t>(pts.size());
  uint32_t* d_rho = ar.take<uint32_t>(rho.size());
  G1Affine* d_key1 = ar.take<G1Affine>(2);
  G2Affine* d_key2 = ar.take<G2Affine>(6);
  G1Affine* d_pt1 = ar.take<G1Affine>(7 * (size_t)n);
  G2Affine* d_pt2 = ar.take<G2Affine>(n);
  uint8_t* d_st = ar.take<uint8_t>(8 * (size_t)n);
  G1XYZZ* d_wg1 = ar.take<G1XYZZ>(PV_G1_ITEMS * (size_t)n);
  G2XYZZ* d_wg2 = ar.take<G2XYZZ>(PV_G2_ITEMS * (size_t)n);
  Fr* d_w1 = ar.take<Fr>(n);
  uint8_t* d_valid = ar.take<uint8_t>(n);
  G1XYZZ* d_Lv = ar.take<G1XYZZ>(n);
  G2XYZZ* d_Lw = ar.take<G2XYZZ>(n);
  G1XYZZ* d_gv = ar.take<G1XYZZ>(P);
  G2XYZZ* d_gw = ar.take<G2XYZZ>(P);
  G1Affine* d_gva = ar.take<G1Affine>(P);
  G2Affine* d_gwa = ar.take<G2Affine>(P);
  Fp12* d_f = ar.take<Fp12>(2 * P);
  G1XYZZ* d_s1 = ar.take<G1XYZZ>((size_t)PV_SUMS1 * 2 * P);
  G2XYZZ* d_s2 = ar.take<G2XYZZ>((size_t)PV_SUMS2 * 2 * P);
  Fp12* d_fe = ar.take<Fp12>(2 * P);
  uint8_t* d_bad = ar.take<uint8_t>(2 * P);
  uint32_t* d_err = ar.take<uint32_t>(1);    // key points; proof points report per proof
  uint32_t* d_perr = ar.take<uint32_t>(1);
  if (!d_key || !d_pts || !d_rho || !d_key1 || !d_key2 || !d_pt1 || !d_pt2 || !d_st || !d_wg1 || !d_wg2 || !d_w1 || !d_valid ||
      !d_Lv || !d_Lw || !d_gv || !d_gw || !d_gva || !d_gwa || !d_f || !d_s1 || !d_s2 || !d_fe || !d_bad || !d_err || !d_perr)
    return PS_ERR_ALLOC;
  PS_TRY(ctx_verify_event(ctx, 0));
  PS_TRY(dev_h2d(d_key, key.data(), key.size(), st));
  PS_TRY(dev_h2d(d_pts, pts.data(), pts.size(), st));
  PS_TRY(dev_h2d(d_rho, rho.data(), rho.size() * 4, st));
  PS_TRY(dev_memset(d_err, 0, 4, st));
  PS_TRY(dev_memset(d_bad, 0, 2 * P, st));
  PS_TRY(ctx_verify_event(ctx, 1));
  // key points follow the context's subgroup_check; proof points are untrusted and always checked, with a status each
  const bool sub = ctx->subgroup_check != 0;
  PS_TRY(GroupOps<Fp>::decode(ctx, d_key, 2, PS_FMT_COMPRESSED, d_key1, d_err, sub));
  PS_TRY(GroupOps<Fp2>::decode(ctx, d_key + 96, 6, PS_FMT_COMPRESSED, d_key2, d_err, sub));
  PS_TRY(GroupOps<Fp>::decode(ctx, d_pts, 7 * (size_t)n, PS_FMT_COMPRESSED, d_pt1, d_perr, true, d_st));
  PS_TRY(GroupOps<Fp2>::decode(ctx, d_pts + 7 * 48 * n_proofs, n, PS_FMT_COMPRESSED, d_pt2, d_perr, true, d_st + 7 * n_proofs));
  PS_TRY(ctx_verify_event(ctx, 2));
  PS_LAUNCH(PvWeighG1K, st, PV_G1_ITEMS * (size_t)n, n, (const uint32_t*)d_rho, (const uint8_t*)d_st, (const G1Affine*)d_pt1, d_wg1);
  PS_LAUNCH(PvWeighG2K, st, PV_G2_ITEMS * (size_t)n, n, (const uint32_t*)d_rho, (const uint8_t*)d_st, (const G2Affine*)d_pt2, d_wg2);
  PS_LAUNCH(PvLeafK, st, P, n, P, (const uint32_t*)d_rho, (const uint8_t*)d_st, (const G1XYZZ*)d_wg1, (const G2XYZZ*)d_wg2, d_s1,
            d_s2, d_w1, d_valid);
  PS_TRY(ctx_verify_event(ctx, 3));
  // per-proof io sums: rho_i1 gv_i over vs (rows rho_i1 io_ik, standard form) and gw_i over ws (rows io_ik, Montgomery)
  uint32_t *d_io = nullptr, *d_ioerr = nullptr;
  if (n_io) {
    PS_TRY(stage_scalars(ctx, io_be, n_proofs * n_io, 1, &d_io, &d_ioerr));
    std::vector<uint32_t> leaves(n);
    for (uint32_t i = 0; i < n; i++) leaves[i] = P + i;
    uint32_t* d_leaves = ar.take<uint32_t>(n);
    Fr* d_rows = ar.take<Fr>(n_proofs * n_io);
    if (!d_leaves || !d_rows) return PS_ERR_ALLOC;
    PS_TRY(dev_h2d(d_leaves, leaves.data(), 4 * (size_t)n, st));
    PS_LAUNCH(VbIoCombineK, st, n_proofs * n_io, (uint32_t)n_io, P, n, (const uint32_t*)d_leaves, (const Fr*)d_io, (const Fr*)d_w1,
              d_rows);
    PS_TRY(msm_rows<Fp>(ctx, bv, (const uint32_t*)d_rows, n, 0, d_Lv));
    PS_TRY(msm_rows<Fp2>(ctx, bw, (const uint32_t*)d_io, n, 1, d_Lw));
  } else {
    PS_TRY(dev_memset(d_Lv, 0, n * sizeof(G1XYZZ), st));
    PS_TRY(dev_memset(d_Lw, 0, n * sizeof(G2XYZZ), st));
  }
  PS_LAUNCH(PvCommitK, st, P, n, (const uint8_t*)d_st, (const G1XYZZ*)d_Lv, (const G2XYZZ*)d_Lw, (const G1XYZZ*)d_wg1, (const G2Affine*)d_pt2, d_gv, d_gw);
  PS_TRY(GroupOps<Fp>::to_affine(ctx, d_gv, P, d_gva));
  PS_TRY(GroupOps<Fp2>::to_affine(ctx, d_gw, P, d_gwa));
  PvState pv{ctx, by, n, P, (uint32_t)n_io, (const Fr*)d_io, d_w1, d_f, d_s1, d_s2, d_fe, d_bad, d_key1, d_key2};
  PS_TRY(ctx_verify_event(ctx, 4));
  PS_LAUNCH(PairingMillerK, st, P, (const G1Affine*)d_gva, (const G2Affine*)d_gwa, d_f + P);
  PS_TRY(ctx_verify_event(ctx, 5));
  for (uint32_t first = P >> 1; first >= 1; first >>= 1) PS_LAUNCH(PvTreeLevelK, st, first, first, P, d_f, d_s1, d_s2);
  PS_TRY(ctx_verify_event(ctx, 6));
  PS_TRY(pv.check_nodes(std::vector<uint32_t>{1}));
  PS_TRY(ctx_verify_event(ctx, 7));
  std::vector<uint8_t> valid(n_proofs);
  uint8_t root_bad = 0;
  PS_TRY(dev_d2h(valid.data(), d_valid, n_proofs, st));
  PS_TRY(dev_d2h(&root_bad, d_bad + 1, 1, st));
  uint32_t herr[2] = {0, 0};
  PS_TRY(dev_d2h(herr, d_err, 4, st));
  if (n_io) PS_TRY(dev_d2h(herr + 1, d_ioerr, 4, st));
  PS_TRY(dev_sync(st));
  if (herr[0] || herr[1]) return PS_ERR_ENCODING;
  bool all_valid = true;
  for (size_t i = 0; i < n_proofs; i++) all_valid = all_valid && valid[i];
  *ok = (all_valid && !root_bad) ? 1 : 0;
  if (per_proof) {
    memcpy(per_proof, valid.data(), n_proofs);
    PS_TRY(bisect(pv, ctx, P, n, d_bad, root_bad != 0, per_proof));
  }
  PS_TRY(ctx_verify_event(ctx, 8));
  ctx->evv_valid = true;
  return PS_OK;
}

}  // extern "C"
