// Kernels of the batch PHGR13 verifier (ps_phgr13_verify_batch, capi_verify.cu).  Proof i gets five independent weights
// rho_i1..rho_i5, one per equation of pinochio.go:312-372 (division, three CRS checks, linear check), and N proofs are
// decided as ONE pairing-product check:
//   prod_i e(rho1 gv_i, gw_i) * e(X - sum_k (sum_i rho_i1 io_ik) ys_k, G2gen) * e(-Hs, yts) e(-Vs, av) e(-Ys, ay)
//   * e(Gz, gamma) e(-VYs, bgamma2) e(-aw, W3) e(-bgamma, W5) == 1,
//   X = sum_i [rho2 vass_i + rho3 wass_i + rho4 yass_i - rho1 yss_i],  Hs = sum rho1 hs_i,  Vs = sum rho2 vss_i,
//   Ys = sum rho4 yss_i,  Gz = sum rho5 gz_i,  VYs = sum rho5 (vss_i + yss_i),  W3 = sum rho3 wss_i,  W5 = sum rho5 wss_i.
// The division check pairs two proof-dependent points, so each proof keeps its own Miller value e(rho1 gv_i, gw_i); its
// io sums gv_i and gw_i are one MSM row each (msm_rows in G1 and G2).  The proofs are the leaves of the same heap-numbered
// tree as the Groth16 batch (verify_batch.cuh): every node keeps its Miller-value product and the eight sums above over
// its proofs, and the node check adds one ys MSM row, eight fixed Miller loops and one final exponentiation.
#pragma once
#include "verify_batch.cuh"

namespace ps {

// proof point layout after decoding: G1 point j of proof i at pt1[j * n + i], j = hs vss yss vass wass yass gz; wss at
// pt2[i]; decode status st[j * n + i] for the G1 points and st[7 n + i] for wss
enum { PV_HS, PV_VSS, PV_YSS, PV_VASS, PV_WASS, PV_YASS, PV_GZ };
constexpr int PV_G1_ITEMS = 10, PV_G2_ITEMS = 2, PV_SUMS1 = 6, PV_SUMS2 = 2;

PS_DEV bool pv_valid(const uint8_t* st, uint32_t n, uint32_t i) {
  uint8_t s = 0;
  for (int j = 0; j < 8; j++) s |= st[(size_t)j * n + i];
  return s == 0;
}

// Weighted G1 points (thread per (item j, proof i)): out[j n + i] = rho_{i,e} * point, 0 for a proof that did not decode.
//   j: 0 rho1 hs, 1 rho1 yss, 2 rho1 vss, 3 rho2 vass, 4 rho2 vss, 5 rho3 wass, 6 rho4 yass, 7 rho4 yss, 8 rho5 gz,
//      9 rho5 (vss + yss)
struct PvWeighG1K {
  static constexpr int BLOCK = 64;
  PS_DEV static void run(uint32_t tid, uint32_t n, const uint32_t* rho, const uint8_t* st, const G1Affine* pt1, G1XYZZ* out) {
    const uint8_t PT[PV_G1_ITEMS] = {PV_HS, PV_YSS, PV_VSS, PV_VASS, PV_VSS, PV_WASS, PV_YASS, PV_YSS, PV_GZ, PV_VSS};
    const uint8_t EQ[PV_G1_ITEMS] = {0, 0, 0, 1, 1, 2, 3, 3, 4, 4};
    const uint32_t j = tid / n, i = tid % n;
    G1XYZZ r = G1XYZZ::inf();
    if (pv_valid(st, n, i)) {
      G1XYZZ base = G1XYZZ::from_affine(pt1[(size_t)PT[j] * n + i]);
      if (j == 9) xyzz_add_c(base, G1XYZZ::from_affine(pt1[(size_t)PV_YSS * n + i]));
      r = xyzz_scalar_mul(base, rho + ((size_t)i * 5 + EQ[j]) * 4, 4);
    }
    out[tid] = r;
  }
};
// Weighted wss (thread per (item j, proof i)): j = 0 rho3 wss, 1 rho5 wss
struct PvWeighG2K {
  static constexpr int BLOCK = 32;
  PS_DEV static void run(uint32_t tid, uint32_t n, const uint32_t* rho, const uint8_t* st, const G2Affine* pt2, G2XYZZ* out) {
    const uint32_t j = tid / n, i = tid % n;
    G2XYZZ r = G2XYZZ::inf();
    if (pv_valid(st, n, i)) r = xyzz_scalar_mul(G2XYZZ::from_affine(pt2[i]), rho + ((size_t)i * 5 + (j == 0 ? 2 : 4)) * 4, 4);
    out[tid] = r;
  }
};

// Leaf values (thread per slot i < P): the node sums of proof i at index P + i of s1 (PV_SUMS1 rows of 2P: X, Hs, Vs, Ys,
// Gz, VYs) and s2 (W3, W5); w1[i] = rho_i1 (0 for a proof that did not decode), valid[i].  Slots i >= n are empty.
struct PvLeafK {
  static constexpr int BLOCK = 64;
  PS_DEV static void run(uint32_t i, uint32_t n, uint32_t P, const uint32_t* rho, const uint8_t* st, const G1XYZZ* wg1,
                         const G2XYZZ* wg2, G1XYZZ* s1, G2XYZZ* s2, Fr* w1, uint8_t* valid) {
    G1XYZZ v[PV_SUMS1];
    G2XYZZ u[PV_SUMS2];
    for (int s = 0; s < PV_SUMS1; s++) v[s] = G1XYZZ::inf();
    for (int s = 0; s < PV_SUMS2; s++) u[s] = G2XYZZ::inf();
    if (i < n) {
      const bool ok = pv_valid(st, n, i);
      auto w = [&](int j) { return wg1[(size_t)j * n + i]; };
      v[0] = w(3);
      xyzz_add_c(v[0], w(5));
      xyzz_add_c(v[0], w(6));
      xyzz_add_c(v[0], w(1).neg());
      v[1] = w(0); v[2] = w(4); v[3] = w(7); v[4] = w(8); v[5] = w(9);
      u[0] = wg2[i]; u[1] = wg2[n + i];
      Fr r1 = Fr::zero();
      if (ok)
        for (int j = 0; j < 4; j++) r1.v[j] = rho[(size_t)i * 20 + j];
      w1[i] = r1;
      valid[i] = ok ? 1 : 0;
    }
    for (int s = 0; s < PV_SUMS1; s++) s1[(size_t)s * 2 * P + P + i] = v[s];
    for (int s = 0; s < PV_SUMS2; s++) s2[(size_t)s * 2 * P + P + i] = u[s];
  }
};

// Operands of the division-check pair of each slot (thread per slot i < P): gv[i] = rho1 gv_i = Lv[i] + rho1 vss_i,
// gw[i] = gw_i = Lw[i] + wss_i, where Lv / Lw are the io MSM rows; an empty slot, and a proof that did not decode, pairs
// infinity with infinity (Miller value 1), so no undecoded point reaches the field arithmetic.
struct PvCommitK {
  static constexpr int BLOCK = 32;
  PS_DEV static void run(uint32_t i, uint32_t n, const uint8_t* st, const G1XYZZ* Lv, const G2XYZZ* Lw, const G1XYZZ* wg1,
                         const G2Affine* pt2, G1XYZZ* gv, G2XYZZ* gw) {
    G1XYZZ a = G1XYZZ::inf();
    G2XYZZ b = G2XYZZ::inf();
    if (i < n && pv_valid(st, n, i)) {
      a = Lv[i];
      xyzz_add_c(a, wg1[(size_t)2 * n + i]);
      b = Lw[i];
      xyzz_add_c(b, G2XYZZ::from_affine(pt2[i]));
    }
    gv[i] = a;
    gw[i] = b;
  }
};

// One level of the tree (thread per node k in [first, 2 first)): Miller-value products and the eight sums
struct PvTreeLevelK {
  static constexpr int BLOCK = 32;
  PS_DEV static void run(uint32_t t, uint32_t first, uint32_t P, Fp12* f, G1XYZZ* s1, G2XYZZ* s2) {
    const uint32_t k = first + t;
    f[k] = fp12_mul(f[2 * k], f[2 * k + 1]);
    for (int s = 0; s < PV_SUMS1; s++) {
      G1XYZZ* row = s1 + (size_t)s * 2 * P;
      G1XYZZ c = row[2 * k];
      xyzz_add_c(c, row[2 * k + 1]);
      row[k] = c;
    }
    for (int s = 0; s < PV_SUMS2; s++) {
      G2XYZZ* row = s2 + (size_t)s * 2 * P;
      G2XYZZ c = row[2 * k];
      xyzz_add_c(c, row[2 * k + 1]);
      row[k] = c;
    }
  }
};

// The eight fixed pairs of each listed node k = nodes[t] (Lio[t] = the node's ys MSM row):
//   (X - Lio, G2gen) (-Hs, yts) (-Vs, av) (-Ys, ay) (Gz, gamma) (-VYs, bgamma2) (-aw, W3) (-bgamma, W5)
// key1 = aw, bgamma; key2 = av, ay, gamma, bgamma2, yts, G2gen
struct PvNodePointsK {
  static constexpr int BLOCK = 32;
  PS_DEV static void run(uint32_t t, uint32_t P, const uint32_t* nodes, const G1XYZZ* s1, const G2XYZZ* s2, const G1XYZZ* Lio,
                         const G1Affine* key1, const G2Affine* key2, G1XYZZ* p, G2XYZZ* q) {
    const uint32_t k = nodes[t];
    auto sum1 = [&](int s) { return s1[(size_t)s * 2 * P + k]; };
    G1XYZZ x = sum1(0);
    xyzz_add_c(x, Lio[t].neg());
    G1XYZZ* pp = p + 8 * (size_t)t;
    G2XYZZ* qq = q + 8 * (size_t)t;
    pp[0] = x;               qq[0] = G2XYZZ::from_affine(key2[5]);
    pp[1] = sum1(1).neg();   qq[1] = G2XYZZ::from_affine(key2[4]);
    pp[2] = sum1(2).neg();   qq[2] = G2XYZZ::from_affine(key2[0]);
    pp[3] = sum1(3).neg();   qq[3] = G2XYZZ::from_affine(key2[1]);
    pp[4] = sum1(4);         qq[4] = G2XYZZ::from_affine(key2[2]);
    pp[5] = sum1(5).neg();   qq[5] = G2XYZZ::from_affine(key2[3]);
    pp[6] = G1XYZZ::from_affine(key1[0]).neg();   qq[6] = s2[k];
    pp[7] = G1XYZZ::from_affine(key1[1]).neg();   qq[7] = s2[(size_t)2 * P + k];
  }
};

// acc[t] = f[nodes[t]] * the eight fixed Miller values of node t
struct PvNodeProductK {
  static constexpr int BLOCK = 32;
  PS_DEV static void run(uint32_t t, const uint32_t* nodes, const Fp12* f, const Fp12* fm, Fp12* acc) {
    Fp12 a = f[nodes[t]];
    for (int j = 0; j < 8; j++) a = fp12_mul(a, fm[8 * (size_t)t + j]);
    acc[t] = a;
  }
};

}  // namespace ps
