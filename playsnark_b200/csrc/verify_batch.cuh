// Kernels of the batch Groth16 verifier (ps_g16_verify_batch, capi_verify.cu).  N proofs against one key are decided as
// ONE pairing-product check with random nonzero 128-bit weights rho_i:
//   prod_i e(-rho_i A_i, B_i) * e(S Alpha, Beta2) * e(L, Gamma) * e(Cs, Delta2) == 1,
//   S = sum_i rho_i,  L = sum_j (sum_i rho_i io_i[j]) IoLP_j,  Cs = sum_i rho_i C_i.
// The proofs are the leaves of a complete binary tree over P = 2^ceil(log2 N) slots, heap-numbered: the root is node 1,
// node k has children 2k and 2k+1, proof i is node P + i.  Every node keeps the product of its proofs' Miller values and
// the sums of their rho_i C_i and rho_i, so the same check restricted to one node's proofs ("node check") costs one io
// MSM, three Miller loops and one final exponentiation.  Because every term is a homomorphism of the node's proof set,
// the check value of node k (after the final exponentiation) is the product of its children's: the per-proof bisection
// computes the left child's value and derives the right one as parent * conj(left) (inverse = conjugate in the
// cyclotomic subgroup).
#pragma once
#include "pairing.cuh"

namespace ps {

// [lo, hi) of the proofs under node k of a tree with P leaves, clipped to n
PS_DEV void vb_node_range(uint32_t k, uint32_t P, uint32_t n, uint32_t& lo, uint32_t& hi) {
  uint32_t d = 0;
  while ((k >> (d + 1)) != 0) d++;               // depth of k
  const uint32_t span = P >> d;
  lo = (k - (1u << d)) * span;
  hi = lo + span < n ? lo + span : n;
  if (lo > hi) lo = hi;
}

// Leaf i (thread per slot, i < P): w_i = rho_i when all three points of proof i decoded into the subgroup, else 0, which
// leaves the proof out of every sum; negA[i] = -w_i A_i, cs[P+i] = w_i C_i, s[P+i] = w_i.  Slots i >= n are empty.
struct VbWeighK {
  static constexpr int BLOCK = 64;
  PS_DEV static void run(uint32_t i, uint32_t n, uint32_t P, const uint32_t* rho, const uint8_t* st, const G1Affine* A,
                         const G1Affine* Cp, G1XYZZ* negA, G1XYZZ* cs, Fr* s, Fr* w, uint8_t* valid) {
    const bool ok = i < n && (st[i] | st[n + i] | st[2 * n + i]) == 0;
    Fr wi = Fr::zero();
    G1XYZZ a = G1XYZZ::inf(), c = G1XYZZ::inf();
    if (ok) {
      const uint32_t* k = rho + (size_t)i * 4;
#pragma unroll
      for (int j = 0; j < 4; j++) wi.v[j] = k[j];
      a = xyzz_scalar_mul(G1XYZZ::from_affine(A[i]), k, 4).neg();
      c = xyzz_scalar_mul(G1XYZZ::from_affine(Cp[i]), k, 4);
    }
    negA[i] = a;
    cs[P + i] = c;
    s[P + i] = wi;
    if (i < n) { w[i] = wi; valid[i] = ok ? 1 : 0; }
  }
};

// One level of the tree (thread per node k in [first, 2 first)): products of Miller values, sums of w_i C_i and of w_i
struct VbTreeLevelK {
  static constexpr int BLOCK = 32;
  PS_DEV static void run(uint32_t t, uint32_t first, Fp12* f, G1XYZZ* cs, Fr* s) {
    const uint32_t k = first + t;
    f[k] = fp12_mul(f[2 * k], f[2 * k + 1]);
    G1XYZZ c = cs[2 * k];
    xyzz_add_c(c, cs[2 * k + 1]);
    cs[k] = c;
    s[k] = s[2 * k] + s[2 * k + 1];
  }
};

// Combined public inputs of the listed nodes (thread per (node t, input j)):
//   out[t][j] = sum over the node's proofs i of io[i][j] * w_i   (io Montgomery, w standard -> the product is standard)
struct VbIoCombineK {
  static constexpr int BLOCK = 128;
  PS_DEV static void run(uint32_t tid, uint32_t n_io, uint32_t P, uint32_t n, const uint32_t* nodes, const Fr* io, const Fr* w,
                         Fr* out) {
    const uint32_t t = tid / n_io, j = tid % n_io;
    uint32_t lo, hi;
    vb_node_range(nodes[t], P, n, lo, hi);
    Fr acc = Fr::zero();
    for (uint32_t i = lo; i < hi; i++) acc = acc + fe_mul_call(io[(size_t)i * n_io + j], w[i]);
    out[tid] = acc;
  }
};

// G1 / G2 operands of the three fixed pairs of each listed node: (S_k Alpha, Beta2), (L_k, Gamma), (Cs_k, Delta2)
struct VbNodePointsK {
  static constexpr int BLOCK = 32;
  PS_DEV static void run(uint32_t t, const uint32_t* nodes, const Fr* s, const G1XYZZ* cs, const G1XYZZ* L, const G1Affine* alpha,
                         const G2Affine* key2, G1XYZZ* p, G2Affine* q) {
    const uint32_t k = nodes[t];
    p[3 * t] = xyzz_scalar_mul(G1XYZZ::from_affine(*alpha), s[k].v, 8);
    p[3 * t + 1] = L[t];
    p[3 * t + 2] = cs[k];
    q[3 * t] = key2[0];
    q[3 * t + 1] = key2[1];
    q[3 * t + 2] = key2[2];
  }
};

// Node check of the listed node k = nodes[t], in two kernels: acc[t] = f[k] * the three fixed Miller values, then
// val[t] = acc[t]^(3 (p^12 - 1) / r)
struct VbNodeProductK {
  static constexpr int BLOCK = 32;
  PS_DEV static void run(uint32_t t, const uint32_t* nodes, const Fp12* f, const Fp12* fm, Fp12* acc) {
    acc[t] = fp12_mul(fp12_mul(f[nodes[t]], fm[3 * t]), fp12_mul(fm[3 * t + 1], fm[3 * t + 2]));
  }
};
struct VbFinalExpK {
  static constexpr int BLOCK = 32;
  PS_DEV static void run(uint32_t t, const Fp12* acc, Fp12* val) { val[t] = final_exponentiation(acc[t]); }
};
// Verdicts of the listed nodes: fe[k] = val[t], bad[k] = fe[k] != 1.  Listed nodes k > 1 are left children: the right
// sibling's value is parent * conj(left), without a check of its own.
struct VbVerdictK {
  static constexpr int BLOCK = 32;
  PS_DEV static void run(uint32_t t, const uint32_t* nodes, const Fp12* val, Fp12* fe, uint8_t* bad) {
    const uint32_t k = nodes[t];
    fe[k] = val[t];
    bad[k] = val[t] == Fp12::one() ? 0 : 1;
    if (k > 1) {
      const Fp12 r = fp12_mul(fe[k >> 1], fp12_conj(val[t]));
      fe[k + 1] = r;
      bad[k + 1] = r == Fp12::one() ? 0 : 1;
    }
  }
};

}  // namespace ps
